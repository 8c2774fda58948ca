"""Generate tests/golden/feed.json by running the UNMODIFIED reference loader code (dataset/pretrain_dataset.py of the original
XFM sources: TextMaskingGenerator, ImageTextJsonDataset.preprocess / collate_fn, TextJsonDataset.preprocess,
RegionTextJsonDataset.__iter__ / get_image_attns / collate_fn) on seeded inputs with the stub tokenizer of tests/feed_stub.py.
Needs a checkout of those sources, named by XFM_REFERENCE_ROOT; the fixture it writes is what tests/test_feed_cpu.py checks
xfm_b200.feed against.

    XFM_REFERENCE_ROOT=<XFM checkout> python tools/make_golden_feed.py
"""
import base64
import contextlib
import importlib.abc
import importlib.machinery
import io
import json
import os
import random
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
REF_ROOT = os.environ.get("XFM_REFERENCE_ROOT", "")
ABSENT = {"pycocotools", "pycocoevalcap", "skimage", "matplotlib", "ruamel", "h5py", "cv2", "ftfy", "timm"}


class _Stub(types.ModuleType):
    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        return type(k, (), {})


class _Finder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    """Evaluation-only dependencies of dataset/__init__.py that are not in the image import as empty stubs."""

    def find_spec(self, name, path, target=None):
        if name.split(".")[0] in ABSENT:
            return importlib.machinery.ModuleSpec(name, self, is_package=True)

    def create_module(self, spec):
        m = _Stub(spec.name)
        m.__path__ = []
        return m

    def exec_module(self, m):
        pass


def reference_module():
    import transformers  # noqa: F401  (before the stubs exist)
    sys.meta_path.append(_Finder())
    sys.path.insert(0, REF_ROOT)
    with contextlib.redirect_stdout(io.StringIO()):
        import dataset.pretrain_dataset as pd
    return pd


def bare(cls, **attrs):
    """An instance without __init__ (which lists data files on HDFS): only the attributes the methods under test read."""
    o = object.__new__(cls)
    o.__dict__.update(attrs)
    return o


def sentence(rng, n):
    from feed_stub import WORDS
    return " ".join(rng.choice(WORDS) for _ in range(n))


def main():
    import torch
    from PIL import Image
    from feed_stub import StubTokenizer

    pd = reference_module()
    gen = random.Random(1234)            # drives the INPUTS; the code under test draws from the global generator
    out = dict(masker=[], preprocess=[], corpus=[], image_atts=[], region=[], collate=[], region_collate=[])   # + lines, image_text
    quiet = contextlib.redirect_stdout(io.StringIO())

    # ---- TextMaskingGenerator
    for style in ("roberta", "bert"):
        tok = StubTokenizer(style)
        for (prob, mmax, sprb, ssize, whole, use_rob) in [(0.25, 8, 0.2, 3, False, False), (0.4, 6, 0.5, 3, True, style == "roberta"),
                                                          (0.15, 4, 0.0, 3, True, style == "roberta"), (0.5, 10, 1.0, 2, False, False)]:
            with quiet:
                mg = pd.TextMaskingGenerator(tok, prob, mmax, sprb, ssize, whole, use_roberta=use_rob)
            for seed in range(6):
                tokens = [tok.cls_token] + tok.tokenize(sentence(gen, gen.randint(1, 9))) + [tok.sep_token]
                random.seed(seed)
                got, pos = mg(list(tokens))
                out["masker"].append(dict(style=style, cfg=[prob, mmax, sprb, ssize, whole, use_rob], seed=seed, tokens=tokens,
                                          tokens_masked=got, masked_pos=pos, next_random=random.random()))

    # ---- preprocess (image-text stream, pretrain_dataset.py:264-300) and the text-only stream (:690-726)
    for style in ("roberta", "bert"):
        tok = StubTokenizer(style)
        with quiet:
            mg = pd.TextMaskingGenerator(tok, 0.25, 5, 0.2, 3, style == "bert")
        for tokenized, lang in [(False, None), (True, None), (False, "zh")]:
            ds = bare(pd.ImageTextJsonDataset, tokenized=tokenized, language_chosen=lang, max_words=7, max_tokens=12, max_masks=5,
                      tokenizer=tok, cls_token=tok.cls_token, eos_token=tok.sep_token, pad_token_id=tok.pad_token_id,
                      add_eos=True, mask_generator=mg, PAD_mask=-100)
            for seed in range(4):
                text = sentence(gen, gen.randint(1, 10))
                if seed == 1:
                    text = "A Man, riding/holding the-horse!  <person> (left)  " + text
                if tokenized and style == "bert":
                    text = " ".join(tok.tokenize(text))
                random.seed(100 + seed)
                res = ds.preprocess(text)
                out["preprocess"].append(dict(style=style, tokenized=tokenized, lang=lang, seed=100 + seed, text=text,
                                              out=[list(map(int, r)) for r in res]))
        for tokenized in (False, True):
            ds = bare(pd.TextJsonDataset, tokenized=tokenized, max_words=7, max_tokens=12, max_masks=5, tokenizer=tok,
                      cls_token=tok.cls_token, eos_token=tok.sep_token, pad_token_id=tok.pad_token_id, add_eos=True,
                      mask_generator=mg, PAD_mask=-100)
            for seed in range(3):
                text = sentence(gen, gen.randint(1, 14))
                if tokenized:
                    text = " ".join(tok.tokenize(text))
                random.seed(200 + seed)
                res = ds.preprocess(text)
                out["corpus"].append(dict(style=style, tokenized=tokenized, seed=200 + seed, text=text,
                                          out=[list(map(int, r)) for r in res]))

    # ---- get_image_attns
    for ps, res in [(16, 224), (16, 384), (32, 224)]:
        ds = bare(pd.RegionTextJsonDataset, patch_size=ps, num_patch=res // ps)
        for _ in range(12):
            x, y = gen.uniform(0, res), gen.uniform(0, res)
            w, h = gen.uniform(0.01, res - x + 3), gen.uniform(0.01, res - y + 3)
            out["image_atts"].append(dict(patch_size=ps, num_patch=res // ps, box=[x, y, w, h],
                                          atts=ds.get_image_attns(x, y, w, h)))
        for box in ([0, 0, res, res], [res - 1e-3, res - 1e-3, 5.0, 5.0], [16.0, 32.0, 16.0, 16.0], [15.999, 0.0, 0.002, 1.0]):
            out["image_atts"].append(dict(patch_size=ps, num_patch=res // ps, box=list(box), atts=ds.get_image_attns(*box)))

    # ---- RegionTextJsonDataset.__iter__ (one annotated image -> region samples) and collate_fn
    tok = StubTokenizer("roberta")
    with quiet:
        mg = pd.TextMaskingGenerator(tok, 0.25, 4, 0.2, 3, False)

    def make_ann(W, H, n_elems, with_caption, multilingual=False):
        buf = io.BytesIO()
        Image.new("RGB", (W, H), (gen.randrange(256), gen.randrange(256), gen.randrange(256))).save(buf, format="PNG")
        elems = []
        for _ in range(n_elems):
            x, y = gen.randrange(0, W - 8), gen.randrange(0, H - 8)
            w, h = gen.randrange(4, W - x + 1), gen.randrange(4, H - y + 1)
            cap = sentence(gen, gen.randint(1, 6))
            e = dict(bb=[x, y, w, h], caption=[cap, sentence(gen, 3)] if gen.random() < 0.4 else cap)
            if gen.random() < 0.4:
                e["attributes"] = [sentence(gen, 1), sentence(gen, 2)]
            elems.append(e)
        ann = dict(binary=base64.b64encode(buf.getvalue()).decode(), elems=elems, size=[W, H])
        if with_caption:
            ann["caption"] = dict(en=sentence(gen, 5), de=sentence(gen, 4)) if multilingual else sentence(gen, 6)
        return ann

    region_samples = []
    for case, (careful, max_regions, min_perc, lang) in enumerate([(False, 5, 0.5, None), (True, 3, 0.2, None), (True, 8, 0.7, "en")]):
        ds = bare(pd.RegionTextJsonDataset, image_key="binary", is_image_rpath=False, caption_key="caption", careful_hflip=careful,
                  max_regions=max_regions, min_perc_in_image=min_perc, box_transform=lambda im: torch.zeros(3, 2, 2),
                  tokenized=False, language_chosen=lang, max_words=7, max_tokens=10, max_masks=4, tokenizer=tok,
                  cls_token=tok.cls_token, eos_token=tok.sep_token, pad_token_id=tok.pad_token_id, add_eos=True, mask_generator=mg,
                  PAD_mask=-100, image_res=224, patch_size=16, num_patch=14, print_broken_data=True, batch_size=6)
        for seed in range(5):
            ann = make_ann(gen.randrange(40, 400), gen.randrange(40, 400), gen.randint(1, 7), gen.random() < 0.6,
                           multilingual=gen.random() < 0.3)
            ds.generate = lambda ann=ann: iter([json.dumps(ann)])
            random.seed(300 + seed)
            (sample,) = list(ds)
            region_samples.append(sample)
            lists = [[list(map(int, r)) for r in col] for col in sample[1:7]]
            ann_in = {k: v for k, v in ann.items() if k != "binary"}
            out["region"].append(dict(cfg=[careful, max_regions, min_perc, lang], seed=300 + seed, ann=ann_in,
                                      n_images=len(sample[0]), lists=lists, target_bbox=[t.tolist() for t in sample[7]],
                                      is_image=list(sample[8]), next_random=random.random()))
    # collate: sub-sampling, padding by re-sampling and padding by repetition
    for seed, (idxs, bs) in enumerate([(list(range(0, 5)), 6), (list(range(5, 10)), 16), (list(range(10, 12)), 40),
                                       (list(range(3, 15, 2)), 9), (list(range(15)), 12)]):
        ds.batch_size = bs
        group = [region_samples[i] for i in idxs]
        assert any(len(s[1]) for s in group)
        random.seed(400 + seed)
        with quiet:
            bt = ds.collate_fn(group)
        out["region_collate"].append(dict(seed=400 + seed, samples=idxs, batch_size=bs, images_shape=list(bt[0].shape),
                                          tensors=[t.tolist() for t in bt[1:]], next_random=random.random()))

    # ---- DistLineReadingDataset.generate (dist_dataset.py:44-83) on local files: rank / worker shards, in-place shuffles, repeat
    import tempfile
    import itertools
    import dataset.dist_dataset as dd
    tmpd = tempfile.mkdtemp(prefix="feed-lines-")
    names = []
    for i in range(7):
        path = os.path.join(tmpd, f"part-{i:02d}")
        with open(path, "w") as f:
            for j in range(1 + i % 3):
                f.write(f"file{i}-line{j}\n")
        names.append(f"part-{i:02d}")
    open(os.path.join(tmpd, "_SUCCESS"), "w").close()
    out["lines"] = []
    for world, rank, shuffle, repeat, workers, wid in [(1, 0, False, False, 0, 0), (1, 0, True, True, 0, 0), (2, 0, True, False, 0, 0),
                                                       (2, 1, True, True, 0, 0), (3, 2, False, False, 2, 1), (2, 1, True, True, 2, 0),
                                                       (7, 3, True, False, 0, 0)]:
        files = sorted(os.path.join(tmpd, n) for n in os.listdir(tmpd))
        ds = object.__new__(dd.DistLineReadingDataset)
        ds.__dict__.update(shuffle=shuffle, rank=rank, world_size=world, repeat=repeat,
                           files=[f for f in files if f.find("_SUCCESS") < 0])
        info = types.SimpleNamespace(id=wid, num_workers=workers) if workers else None
        orig = torch.utils.data.get_worker_info
        torch.utils.data.get_worker_info = lambda info=info: info
        try:
            random.seed(500 + world + rank)
            with quiet:
                got = list(itertools.islice(ds.generate(), 40))
        finally:
            torch.utils.data.get_worker_info = orig
        out["lines"].append(dict(world=world, rank=rank, shuffle=shuffle, repeat=repeat, workers=workers, worker_id=wid,
                                 seed=500 + world + rank, names=names, lines=got, next_random=random.random()))
    out["line_files"] = {n: open(os.path.join(tmpd, n)).read() for n in names}

    # ---- ImageTextJsonDataset.__iter__ (:225-262) and ImageJsonDataset.__iter__ (:368-394)
    def png(w, h, rgb):
        buf = io.BytesIO()
        Image.new("RGB", (w, h), rgb).save(buf, format="PNG")
        return base64.b64encode(buf.getvalue()).decode()

    def probe(im):      # which image was decoded (no random draws inside the transform)
        return torch.tensor([im.size[0], im.size[1], *im.getpixel((0, 0))])

    tok = StubTokenizer("roberta")
    with quiet:
        mg = pd.TextMaskingGenerator(tok, 0.25, 4, 0.2, 3, False)
    lines = []
    for i in range(10):
        imgs = [png(2 + gen.randrange(5), 2 + gen.randrange(5), (gen.randrange(256), gen.randrange(256), gen.randrange(256)))
                for _ in range(1 + gen.randrange(3))]
        cap = sentence(gen, gen.randint(1, 6))
        kind = i % 5
        ann = dict(binary=imgs[0] if kind in (0, 3) else imgs,
                   desc=[cap, sentence(gen, 2)] if kind == 1 else dict(en=cap, fr=sentence(gen, 3)) if kind == 2 else cap)
        lines.append(json.dumps(ann))
    lines.insert(3, json.dumps(dict(binary=[], desc="a dog")))                  # no image: skipped silently
    lines.insert(5, json.dumps(dict(binary=png(3, 3, (1, 2, 3)), desc="")))      # empty caption: broken sample
    lines.insert(7, "{not json")                                                  # broken line
    lines.insert(8, json.dumps(["a", "list"]))                                    # not a dict
    out["image_text"] = []
    for lang, text_stream in [(None, True), ("en", True), (None, False)]:
        cls = pd.ImageTextJsonDataset if text_stream else pd.ImageJsonDataset
        ds = bare(cls, image_key="binary", is_image_rpath=False, caption_key="desc", tokenized=False, language_chosen=lang,
                  max_words=7, max_tokens=10, max_masks=4, tokenizer=tok, cls_token=tok.cls_token, eos_token=tok.sep_token,
                  pad_token_id=tok.pad_token_id, add_eos=True, mask_generator=mg, PAD_mask=-100, transform=probe,
                  print_broken_data=False, prefix=['A image of ', 'The image contains ', 'We can see ', 'A picture of '])
        use = [l for l in lines if lang is None or '"fr"' in l or '"desc": "' in l or not l.startswith("{\"binary")]
        ds.generate = lambda use=use: iter(use)
        random.seed(600)
        samples = list(ds)
        out["image_text"].append(dict(lang=lang, text=text_stream, seed=600, lines=use,
                                      samples=[[s[0].tolist()] + [None if v is None else list(map(int, v)) for v in s[1:]]
                                               for s in samples], next_random=random.random()))

    # ---- ImageTextJsonDataset.collate_fn
    ds = bare(pd.ImageTextJsonDataset)
    batch = [(torch.full((3, 2, 2), float(i)), [i, 1, 2], [1, 1, 0], None) for i in range(4)]
    bt = ds.collate_fn(batch)
    out["collate"].append(dict(image=bt[0].tolist(), ids=bt[1].tolist(), atts=bt[2].tolist(), none=bt[3]))

    # ---- fine-tuning loaders: re_train_dataset / re_eval_dataset / nlvr_dataset / vqa_dataset sample logic
    import dataset.retrieval_dataset as rd
    import dataset.nlvr_dataset  # noqa: F401  (the package attribute of the same name is the class: take the modules from sys.modules)
    import dataset.vqa_dataset  # noqa: F401
    nd, vd = sys.modules["dataset.nlvr_dataset"], sys.modules["dataset.vqa_dataset"]
    import dataset.utils as du
    tmpd2 = tempfile.mkdtemp(prefix="feed-ft-")
    Image.new("RGB", (8, 6), (10, 20, 30)).save(os.path.join(tmpd2, "a.png"))
    ids = [gen.choice(["coco_7", "coco_3", 11, "coco_9", 5]) for _ in range(14)]
    train_anns = [dict(image="a.png", image_id=i, caption=sentence(gen, 4)) for i in ids]
    f1 = os.path.join(tmpd2, "train.json")
    json.dump(train_anns, open(f1, "w"))
    ds = rd.re_train_dataset([f1], lambda im: torch.zeros(1), tmpd2)
    got = [ds[i] for i in range(len(ds))]
    eval_anns = [dict(image=f"img{i}.png", caption=["A Dog, on the-left!  " + sentence(gen, gen.randint(2, 40)) for _ in range(1 + i % 3)])
                 for i in range(6)]
    f2 = os.path.join(tmpd2, "eval.json")
    json.dump(eval_anns, open(f2, "w"))
    es = rd.re_eval_dataset(f2, None, tmpd2)
    out["retrieval"] = [dict(train_anns=train_anns, img_ids=[[k, v] for k, v in ds.img_ids.items()],
                             samples=[[c, i] for _, c, i in got], eval_anns=eval_anns, text=es.text, image=es.image,
                             txt2img=[[k, v] for k, v in es.txt2img.items()], img2txt=[[k, v] for k, v in es.img2txt.items()])]
    nl = [dict(images=["a.png", "a.png"], sentence="The LEFT image: two dogs/cats, (maybe)  " + sentence(gen, 35), label=l)
          for l in ("True", "False", "True")]
    f3 = os.path.join(tmpd2, "nlvr.json")
    json.dump(nl, open(f3, "w"))
    ns = nd.nlvr_dataset([f3], lambda im: torch.zeros(1), tmpd2)
    out["nlvr"] = [dict(anns=nl, samples=[[ns[i][2], ns[i][3]] for i in range(len(ns))])]
    vq = []
    for i in range(12):
        kind = i % 4
        q = ["What is on the LEFT side?", "How many dogs/cats are there, really?", "Is this a wooden-table (or not)?  ",
             "what color is the " + sentence(gen, 40)][kind]
        if kind == 1:
            vq.append(dict(image="a.png", dataset="vg", question=q, answer="two", question_id=i))
        else:
            ans = [gen.choice(["yes", "no", "left", "red", "two"]) for _ in range(10)]
            a = dict(image="a.png", question=q, answer=ans, question_id=i)
            if kind == 2:
                a["dataset"] = "vqa"
            vq.append(a)
    f4 = os.path.join(tmpd2, "vqa.json")
    json.dump(vq, open(f4, "w"))
    flips = []
    orig_hflip = vd.hflip
    vd.hflip = lambda im: (flips.append(True), im)[1]
    orig_tok = vd.build_tokenizer
    vd.build_tokenizer = lambda *_: StubTokenizer("roberta")
    try:
        with quiet:
            vs = vd.vqa_dataset([f4], lambda im: torch.zeros(1), tmpd2, tmpd2, split="train")
        samples = []
        random.seed(700)
        for i in range(len(vs)):
            n0 = len(flips)
            _, q, a, w = vs[i]
            samples.append([len(flips) > n0, q, a, w])
        nxt = random.random()
    finally:
        vd.hflip, vd.build_tokenizer = orig_hflip, orig_tok
    out["vqa"] = [dict(anns=vq, seed=700, samples=samples, next_random=nxt,
                       pre_question=[[q, n, du.pre_question(q, n)] for q in [a["question"] for a in vq] for n in (3, 30, 50)])]

    # ---- scheduler.py create_scheduler: lr of a 2-group optimizer over the whole schedule
    import scheduler as ref_sched
    import utils as ref_utils
    out["scheduler"] = []
    for a in [dict(sched="linear", epochs=3, step_per_epoch=7, num_warmup_steps=0.2), dict(sched="linear", num_training_steps=25, num_warmup_steps=5),
              dict(sched="linear", num_training_steps=10, num_warmup_steps=0), dict(sched="linear", epochs=1, step_per_epoch=4, num_warmup_steps=0.9)]:
        args = ref_utils.AttrDict(dict(a))
        w = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.SGD([dict(params=[w], lr=1e-4), dict(params=[torch.nn.Parameter(torch.zeros(1))], lr=2e-4)], lr=1e-4)
        with quiet:
            sch = ref_sched.create_scheduler(args, opt)
        lrs = []
        for _ in range(args["num_training_steps"] + 3):
            lrs.append([g["lr"] for g in opt.param_groups])
            opt.step()
            sch.step()
        out["scheduler"].append(dict(args=a, resolved=[args["num_training_steps"], args["num_warmup_steps"]], lrs=lrs))

    # ---- dataset/randaugment.py: operation sampling (all 14 operations; the functions replaced by recorders, cv2 is not in the
    # image) and the four look-up-table operations (cv2.split / merge / calcHist stand-ins in numpy: channel views, stacking,
    # a float32 [256, 1] count column — what those calls return)
    import numpy as np
    import dataset.randaugment as ra
    cv2 = sys.modules["cv2"]
    cv2.split = lambda img: [img[:, :, c] for c in range(img.shape[2])]
    cv2.merge = lambda chs: np.stack(chs, axis=2)
    cv2.calcHist = lambda imgs, ch, mask, size, rng_: np.bincount(imgs[0].reshape(-1), minlength=size[0]).astype(np.float32).reshape(-1, 1)
    out["randaugment"] = []
    fired = []
    orig_funcs = dict(ra.func_dict)
    for name in ra.func_dict:
        ra.func_dict[name] = (lambda name: lambda img, *args: (fired.append([name, list(args)]), img)[1])(name)
    try:
        for N, M, augs in [(2, 7, ['Identity', 'AutoContrast', 'Equalize', 'Brightness', 'Sharpness', 'ShearX', 'ShearY', 'TranslateX',
                                   'TranslateY', 'Rotate']), (2, 7, ['Identity', 'AutoContrast', 'Equalize', 'Brightness', 'Sharpness']),
                           (3, 10, []), (1, 3, [])]:
            aug = ra.RandomAugment(N, M, isPIL=True, augs=augs)
            runs = []
            np.random.seed(800 + N + M)
            for _ in range(25):
                del fired[:]
                aug(Image.new("RGB", (4, 4)))
                runs.append([[n, [list(a) if isinstance(a, tuple) else a for a in args]] for n, args in fired])
            out["randaugment"].append(dict(N=N, M=M, augs=augs, seed=800 + N + M, runs=runs, next_random=float(np.random.random())))
    finally:
        ra.func_dict.update(orig_funcs)
    out["randaugment_ops"] = []
    nrng = np.random.default_rng(3)
    for t in range(8):
        img = nrng.integers(0, 256, size=(12, 10, 3), dtype=np.uint8)
        if t == 1:
            img[:, :, 0] = 77                       # a constant channel: high <= low, equalize step 0
        if t == 2:
            img = (img // 4 + 90).astype(np.uint8)  # narrow range
        if t == 3:
            img[:] = nrng.integers(0, 2, size=img.shape) * 255
        res = dict(image=img.tolist(), AutoContrast=ra.autocontrast_func(img).tolist(), Equalize=ra.equalize_func(img).tolist(),
                   Identity=ra.identity_func(img).tolist())
        for f in (0.1, 0.1 + 1.8 * 0.7, 1.9):
            res[f"Brightness:{f!r}"] = ra.brightness_func(img, f).tolist()
        out["randaugment_ops"].append(res)

    # ---- vqa_collate_fn (dataset/__init__.py:200-208)
    import dataset as ref_dataset
    vb = [(torch.full((3, 2, 2), float(i)), f"question {i}", [f"a{i}{j}" for j in range(1 + i % 3)],
           [0.25 * (j + 1) for j in range(1 + i % 3)]) for i in range(5)]
    im, qs, ans, w, n = ref_dataset.vqa_collate_fn(vb)
    out["vqa_collate"] = [dict(image=im.tolist(), questions=qs, answers=ans, weights=w.tolist(), weights_dtype=str(w.dtype), n=n)]

    path = os.path.join(ROOT, "tests", "golden", "feed.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print(path, os.path.getsize(path), "bytes;", {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
