"""Helper for tests/test_feed_cpu.py — run as a SUBPROCESS (it registers import stubs), only where XFM_REFERENCE_ROOT names a
checkout of the original XFM sources.  Differential check on fresh random cases, beyond the committed fixture: the
reference's TextMaskingGenerator / preprocess / get_image_attns / RandomAugment sampling and xfm_b200.feed, same seeds.
Prints one JSON object."""
import contextlib
import io
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import numpy as np
    import make_golden_feed as G
    from feed_stub import StubTokenizer, WORDS
    from xfm_b200 import feed

    pd = G.reference_module()
    import dataset.randaugment as ra
    quiet = contextlib.redirect_stdout(io.StringIO())
    gen = random.Random(int(sys.argv[1]) if len(sys.argv) > 1 else 99)
    res = dict(masker=0, preprocess=0, image_atts=0, randaugment=0, mismatches=[])
    for style in ("roberta", "bert"):
        tok = StubTokenizer(style)
        for _ in range(12):
            cfg = (gen.choice([0.15, 0.25, 0.4, 0.6]), gen.randint(1, 10), gen.choice([0.0, 0.2, 0.7, 1.0]), gen.randint(1, 4),
                   gen.random() < 0.5, style == "roberta" and gen.random() < 0.5)
            with quiet:
                ref = pd.TextMaskingGenerator(tok, *cfg[:5], use_roberta=cfg[5])
            mine = feed.TextMasker(tok, *cfg[:5], use_roberta=cfg[5])
            ds = G.bare(pd.ImageTextJsonDataset, tokenized=False, language_chosen=None, max_words=gen.randint(3, 12),
                        max_tokens=gen.randint(4, 16), max_masks=cfg[1], tokenizer=tok, cls_token=tok.cls_token,
                        eos_token=tok.sep_token, pad_token_id=tok.pad_token_id, add_eos=True, mask_generator=ref, PAD_mask=-100)
            tp = feed.TextPreprocessor(tok, mine, max_tokens=ds.max_tokens, max_masks=cfg[1], max_words=ds.max_words)
            for _ in range(25):
                text = " ".join(gen.choice(WORDS) for _ in range(gen.randint(1, 14)))
                tokens = [tok.cls_token] + tok.tokenize(text) + [tok.sep_token]
                seed = gen.randrange(1 << 30)
                random.seed(seed)
                a = ref(list(tokens)), random.random()
                random.seed(seed)
                b = mine(list(tokens)), random.random()
                res["masker"] += 1
                if a != b:
                    res["mismatches"].append(["masker", style, cfg, seed, tokens])
                random.seed(seed)
                a = [list(map(int, r)) for r in ds.preprocess(text)], random.random()
                random.seed(seed)
                b = [list(r) for r in tp.preprocess(text)], random.random()
                res["preprocess"] += 1
                if a != b:
                    res["mismatches"].append(["preprocess", style, cfg, seed, text])
    for _ in range(400):
        ps = gen.choice([14, 16, 32])
        n = gen.choice([7, 14, 24])
        r = ps * n
        x, y = gen.uniform(0, r), gen.uniform(0, r)
        w, h = gen.uniform(1e-3, r - x + 2), gen.uniform(1e-3, r - y + 2)
        ds = G.bare(pd.RegionTextJsonDataset, patch_size=ps, num_patch=n)
        res["image_atts"] += 1
        if ds.get_image_attns(x, y, w, h) != feed.region_image_atts(x, y, w, h, ps, n):
            res["mismatches"].append(["image_atts", ps, n, x, y, w, h])
    fired = []
    for name in list(ra.func_dict):
        ra.func_dict[name] = (lambda name: lambda img, *args: (fired.append((name, args)), img)[1])(name)
    for _ in range(40):
        N, M = gen.randint(1, 4), gen.randint(0, 10)
        augs = gen.sample(list(feed.RandAugmentSampler.ALL), gen.randint(1, 14)) if gen.random() < 0.7 else []
        seed = gen.randrange(1 << 30)
        aug, mine = ra.RandomAugment(N, M, isPIL=False, augs=augs), feed.RandAugmentSampler(N, M, augs)
        for _ in range(10):
            np.random.seed(seed)
            del fired[:]
            aug(np.zeros((2, 2, 3), np.uint8))
            a = list(fired), float(np.random.random())
            np.random.seed(seed)
            b = mine.sample(), float(np.random.random())
            seed += 1
            res["randaugment"] += 1
            if a != b:
                res["mismatches"].append(["randaugment", N, M, augs, seed - 1])
    res["datasets"] = datasets(pd, G, gen, res["mismatches"])
    res["mismatches"] = res["mismatches"][:5]
    print("PROBE_JSON " + json.dumps(res))


def datasets(pd, G, gen, mismatches):
    """The four dataset classes end to end on JSON-line files written here: the reference's ImageTextJsonDataset /
    ImageJsonDataset / RegionTextJsonDataset / TextJsonDataset (build_tokenizer replaced by the stub tokenizer) against the
    classes of the same names in xfm_b200.feed — every sample of one epoch (shuffled, sharded over ranks) and one collated
    batch, same `random` seed."""
    import base64
    import tempfile
    import torch
    from PIL import Image
    from feed_stub import StubTokenizer, WORDS
    from xfm_b200 import feed

    tok = StubTokenizer("roberta")
    pd.build_tokenizer = lambda *_: tok
    quiet = contextlib.redirect_stdout(io.StringIO())

    def words(n):
        return " ".join(gen.choice(WORDS) for _ in range(n))

    def png(w, h):
        im = Image.new("RGB", (w, h))
        im.putdata([(gen.randrange(256), gen.randrange(256), gen.randrange(256)) for _ in range(w * h)])
        buf = io.BytesIO()
        im.save(buf, format="PNG")
        return base64.b64encode(buf.getvalue()).decode()

    root = tempfile.mkdtemp(prefix="feed-ds-")
    dirs = {}
    for kind in ("pairs", "regions", "texts"):
        d = dirs[kind] = os.path.join(root, kind)
        os.makedirs(d)
        for f in range(4):
            with open(os.path.join(d, f"part-{f}"), "w") as fh:
                for _ in range(5):
                    if kind == "pairs":
                        ann = dict(binary=png(gen.randint(2, 6), gen.randint(2, 6)), desc=gen.choice([words(gen.randint(1, 9)), [words(3), words(5)], ""]))
                    elif kind == "texts":
                        ann = dict(text="  " + words(gen.randint(1, 20)) + " ")
                    else:
                        W, H = gen.randint(30, 90), gen.randint(30, 90)
                        elems = []
                        for _ in range(gen.randint(1, 5)):
                            x, y = gen.randrange(0, W - 8), gen.randrange(0, H - 8)
                            e = dict(bb=[x, y, gen.randrange(4, W - x + 1), gen.randrange(4, H - y + 1)],
                                     caption=gen.choice([words(3), [words(2), "on the left " + words(2)]]))
                            if gen.random() < 0.3:
                                e["attributes"] = [words(1), words(2)]
                            elems.append(e)
                        ann = dict(binary=png(W, H), elems=elems)
                        if gen.random() < 0.5:
                            ann["caption"] = words(4)
                    fh.write(json.dumps(ann) + "\n")
    config = dict(text_encoder="roberta-base", mask_prob=0.25, max_masks=4, skipgram_prb=0.2, skipgram_size=3, mask_whole_word=True,
                  max_words=8, max_tokens=12, image_res=32, patch_size=16, print_broken_data=False,
                  images=dict(image_key="binary", is_image_rpath=False, caption_key="desc", batch_size=3, tokenized=False),
                  regions=dict(image_key="binary", is_image_rpath=False, caption_key="caption", batch_size=7, tokenized=False,
                               max_regions=3, min_perc_in_image=0.3, careful_hflip=True),
                  texts=dict(text_key="text", batch_size=4, tokenized=False, mask_prob=0.3, max_masks=5, mask_whole_word=False,
                             max_words=30, max_tokens=10))

    def pixels(im):
        return torch.tensor(list(im.getdata()), dtype=torch.uint8).reshape(im.size[1], im.size[0], 3)

    def plain(x):
        if isinstance(x, torch.Tensor):
            return x.tolist()
        if isinstance(x, (list, tuple)):
            return [plain(v) for v in x]
        return x

    checked = 0
    for name, d, kw in [("ImageTextJsonDataset", "pairs", dict(transform=lambda im: torch.tensor(im.size))),
                        ("ImageJsonDataset", "pairs", dict(transform=lambda im: torch.tensor(im.size))),
                        ("RegionTextJsonDataset", "regions", dict(transform=None, box_transform=pixels)),
                        ("TextJsonDataset", "texts", {})]:
        for rank, world in [(0, 1), (1, 2), (0, 4)]:
            seed = gen.randrange(1 << 30)
            outs = []
            for side in (pd, feed):
                extra = dict(tokenizer=tok) if side is feed else {}
                with quiet:
                    ds = getattr(side, name)(dict(config, images=dict(config["images"]), regions=dict(config["regions"]), texts=dict(config["texts"])),
                                            dirs[d], rank=rank, world_size=world, shuffle=True, repeat=False, **kw, **extra)
                    random.seed(seed)
                    samples = list(ds)
                    batch = ds.collate_fn(samples[:ds.batch_size]) if name != "RegionTextJsonDataset" else \
                        ds.collate_fn([s for s in samples if len(s[0])][:4])
                outs.append((plain(samples), plain(batch), random.random()))
            checked += len(outs[0][0])
            if outs[0] != outs[1]:
                mismatches.append(["dataset", name, rank, world, seed])
    return checked


if __name__ == "__main__":
    main()
