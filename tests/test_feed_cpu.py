"""Host half of the batch feeder (xfm_b200/feed.py, SURVEY.md §8 f4 loader side) against tests/golden/feed.json, which
tools/make_golden_feed.py wrote by running the unmodified reference loader code (dataset/pretrain_dataset.py) on the same seeded
inputs.  Everything here is integer / index work: the bar is exact equality, including the state of the global `random`
generator afterwards (same number of draws in the same order)."""
import json
import os
import random
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from feed_stub import StubTokenizer  # noqa: E402
from xfm_b200 import feed  # noqa: E402


@pytest.fixture(scope="module")
def golden(golden_dir):
    with open(os.path.join(golden_dir, "feed.json")) as f:
        return json.load(f)


def test_text_masker_matches_reference(golden):
    toks = {s: StubTokenizer(s) for s in ("roberta", "bert")}
    assert len(golden["masker"]) == 48
    hit_trim = hit_random_word = 0
    for g in golden["masker"]:
        prob, mmax, sprb, ssize, whole, use_rob = g["cfg"]
        m = feed.TextMasker(toks[g["style"]], prob, mmax, sprb, ssize, whole, use_roberta=use_rob)
        random.seed(g["seed"])
        got, pos = m(list(g["tokens"]))
        assert got == g["tokens_masked"] and pos == g["masked_pos"], g
        assert random.random() == g["next_random"]      # same number of draws
        assert len(pos) <= mmax and 0 not in pos
        hit_random_word += sum(1 for a, b in zip(got, g["tokens"]) if a != b and a != toks[g["style"]].mask_token)
        hit_trim += len(pos) == min(mmax, max(1, int(round(len(g["tokens"]) * prob))))
    assert hit_random_word > 0 and hit_trim > 0          # the fixture reaches the random-word and the full-budget branches


def test_text_masker_private_generator_and_errors():
    tok = StubTokenizer("roberta")
    tokens = [tok.cls_token] + tok.tokenize("a man riding a horse on the street") + [tok.sep_token]
    a = feed.TextMasker(tok, 0.3, 5, rng=random.Random(5))(list(tokens))
    random.seed(5)
    b = feed.TextMasker(tok, 0.3, 5)(list(tokens))
    assert a == b
    with pytest.raises(AssertionError):
        feed.TextMasker(tok, 0.3, 5)(tokens[1:])
    with pytest.raises(ValueError):
        feed.TextMasker(({0: "a", 2: "b"}, "a", "b"), 0.3, 5)


def test_pre_caption():
    assert feed.pre_caption("A Man, riding/holding the-horse!  <person> (left)\n", 50) == "a man riding holding the horse person left"
    assert feed.pre_caption("one two three four", 2) == "one two"
    with pytest.raises(ValueError):
        feed.pre_caption(" ?! ", 5)


def _text(tok, style, tokenized, lang, corpus=False):
    masker = feed.TextMasker(tok, 0.25, 5, 0.2, 3, style == "bert")
    return feed.TextPreprocessor(tok, masker, max_tokens=12, max_masks=5, max_words=7, tokenized=tokenized, language_chosen=lang,
                                 corpus=corpus)


def test_preprocess_matches_reference(golden):
    toks = {s: StubTokenizer(s) for s in ("roberta", "bert")}
    assert len(golden["preprocess"]) == 24 and len(golden["corpus"]) == 12
    for g in golden["preprocess"]:
        tp = _text(toks[g["style"]], g["style"], g["tokenized"], g["lang"])
        random.seed(g["seed"])
        out = tp.preprocess(g["text"])
        assert [list(o) for o in out] == g["out"], g
        ids, atts, ids_m, pos, mids = out
        assert len(ids) == len(atts) == len(ids_m) == 12 and len(pos) == len(mids) == 5
        assert all(m == -100 or ids[p] == m for p, m in zip(pos, mids))
    for g in golden["corpus"]:
        tp = _text(toks[g["style"]], g["style"], g["tokenized"], None, corpus=True)
        random.seed(g["seed"])
        assert [list(o) for o in tp.preprocess(g["text"])] == g["out"], g


def test_region_image_atts_matches_reference(golden):
    assert len(golden["image_atts"]) == 48
    for g in golden["image_atts"]:
        atts = feed.region_image_atts(*g["box"], g["patch_size"], g["num_patch"])
        assert atts == g["atts"], g["box"]
        assert atts[0] == 1 and sum(atts) >= 2


def _region_sampler(cfg, tok):
    careful, max_regions, min_perc, lang = cfg
    text = feed.TextPreprocessor(tok, feed.TextMasker(tok, 0.25, 4, 0.2, 3, False), max_tokens=10, max_masks=4, max_words=7,
                                 language_chosen=lang)
    return feed.RegionSampler(text, image_res=224, patch_size=16, max_regions=max_regions, min_perc_in_image=min_perc,
                              careful_hflip=careful)


def _region_samples(golden):
    tok = StubTokenizer("roberta")
    samples = []
    for g in golden["region"]:
        rs = _region_sampler(g["cfg"], tok)
        W, H = g["ann"]["size"]
        random.seed(g["seed"])
        plan = rs.plan(g["ann"], W, H)
        sample = rs.finish(g["ann"], plan, torch.zeros(3, 2, 2))
        samples.append((g, plan, sample, random.random()))
    return samples


def test_region_sampler_matches_reference(golden):
    assert len(golden["region"]) == 15
    n_regions = n_full = 0
    for g, plan, sample, nxt in _region_samples(golden):
        W, H = g["ann"]["size"]
        assert 0 <= plan.x0 and 0 <= plan.y0 and plan.x0 + plan.w0 <= W and plan.y0 + plan.h0 <= H
        assert len(sample[0]) == g["n_images"]
        assert [[list(r) for r in col] for col in sample[1:7]] == g["lists"], g["seed"]
        assert [t.tolist() for t in sample[7]] == g["target_bbox"]       # float32 values, exact
        assert list(sample[8]) == g["is_image"]
        assert nxt == g["next_random"]
        n_regions += g["is_image"].count(0)
        n_full += g["is_image"].count(1)
    assert n_regions > 10 and n_full > 3


def test_collate_and_region_collate_match_reference(golden):
    g = golden["collate"][0]
    batch = [(torch.full((3, 2, 2), float(i)), [i, 1, 2], [1, 1, 0], None) for i in range(4)]
    img, ids, atts, none = feed.collate(batch)
    assert img.tolist() == g["image"] and ids.tolist() == g["ids"] and atts.tolist() == g["atts"] and none is None
    assert ids.dtype == torch.int64

    samples = [s for _, _, s, _ in _region_samples(golden)]
    branches = set()
    for g in golden["region_collate"]:
        group = [samples[i] for i in g["samples"]]
        n = sum(len(s[1]) for s in group)
        branches.add("sample" if n >= g["batch_size"] else "pad" if 2 * n >= g["batch_size"] else "repeat")
        random.seed(g["seed"])
        bt = feed.region_collate(group, g["batch_size"], warn=lambda *a, **k: None)
        assert list(bt[0].shape) == g["images_shape"]
        assert [t.tolist() for t in bt[1:]] == g["tensors"], g["seed"]
        assert random.random() == g["next_random"]
        idx = bt[1]
        assert idx.dtype == torch.int64 and idx.numel() == g["batch_size"] and int(idx.max()) < bt[0].shape[0]
        assert bt[7].shape == (g["batch_size"], 197) and bt[8].shape == (g["batch_size"], 4) and bt[8].dtype == torch.float32
    assert branches == {"sample", "pad", "repeat"}


def test_to_uint8_hwc_and_cpu_transform_restatement():
    """`to_uint8_hwc` hands over the pixels untouched, and (u8 / 255 - mean) / std — what tests/test_feed_gpu.py holds the
    kernel to — IS torchvision's ToTensor + Normalize on that crop."""
    np = pytest.importorskip("numpy")
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, size=(32, 24, 3), dtype=np.uint8)
    t = feed.to_uint8_hwc(a)
    assert t.dtype == torch.uint8 and t.shape == (32, 24, 3) and (t.numpy() == a).all()
    with pytest.raises(ValueError):
        feed.to_uint8_hwc(a[:, :, 0])
    tv = pytest.importorskip("torchvision.transforms")
    from PIL import Image
    ref = tv.Compose([tv.ToTensor(), tv.Normalize(feed.CLIP_MEAN, feed.CLIP_STD)])(Image.fromarray(a))
    from oracle.feed_oracle import to_tensor_normalize
    assert torch.equal(to_tensor_normalize(t[None], feed.CLIP_MEAN, feed.CLIP_STD)[0], ref)
    flipped = to_tensor_normalize(t[None], feed.CLIP_MEAN, feed.CLIP_STD, flip=torch.ones(1))[0]
    assert torch.equal(flipped, tv.Compose([tv.RandomHorizontalFlip(1.0), tv.ToTensor(), tv.Normalize(feed.CLIP_MEAN, feed.CLIP_STD)])(Image.fromarray(a)))
    assert (feed.to_uint8_hwc(Image.fromarray(a)) == t).all()


def test_device_feeder_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError):
        feed.DeviceFeeder([])


def _resample_with_taps(img, box, out_h, out_w):
    """xfm_b200.feed's tap tables evaluated the way csrc/feed.cu evaluates them (oracle/feed_oracle.py)."""
    from oracle.feed_oracle import resample_with_taps
    plan = feed.crop_resize_plan([img.shape[:2]], [box], out_h, out_w)
    return resample_with_taps(img, box, *(plan[k][0].numpy() for k in ("hb", "hk", "vb", "vk")))


def test_pillow_bicubic_taps_reproduce_pil_resize():
    """The host half of the GPU crop + resize: tap tables in Pillow's 8.22 fixed point.  Evaluated with integer arithmetic they
    give PIL's `crop(box).resize(size, BICUBIC)` bit for bit (down- and up-scaling, full image, thin crops)."""
    np = pytest.importorskip("numpy")
    from oracle.feed_oracle import pil_crop_resize
    rng = np.random.default_rng(7)
    for t in range(24):
        H, W = int(rng.integers(12, 500)), int(rng.integers(12, 500))
        img = rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
        x0, y0 = int(rng.integers(0, W - 6)), int(rng.integers(0, H - 6))
        box = (x0, y0, int(rng.integers(x0 + 3, W + 1)), int(rng.integers(y0 + 3, H + 1)))
        if t % 4 == 0:
            box = (0, 0, W, H)
        oh, ow = [(224, 224), (384, 384), (32, 48)][t % 3]
        ref = pil_crop_resize(img, box, oh, ow)
        assert (_resample_with_taps(img, box, oh, ow) == ref).all(), (t, (H, W), box, (oh, ow))
    first, count, taps = feed.pillow_bicubic_taps(224, 224)          # same size: the identity
    assert (taps.sum(1) == 1 << 22).all() and ((taps != 0).sum(1) == 1).all()
    assert (first + np.argmax(taps, 1) == np.arange(224)).all()


def test_crop_resize_plan_layout_and_errors():
    plan = feed.crop_resize_plan([(50, 40), (30, 70)], [(0, 0, 40, 50), (10, 5, 70, 25)], 16, 24)
    d = plan["desc"]
    assert d.dtype == torch.int64 and d.shape == (2, 8)
    assert d[0].tolist() == [0, 40, 0, 0, 40, 50, 0, 0] and d[1].tolist() == [50 * 40 * 3, 70, 10, 5, 60, 20, 50 * 24 * 3, 0]
    assert plan["src_bytes"] == (50 * 40 + 30 * 70) * 3 and plan["tmp_bytes"] == (50 + 20) * 24 * 3 and plan["max_rows"] == 50
    assert plan["hb"].shape == (2, 24, 2) and plan["vb"].shape == (2, 16, 2) and plan["hk"].dtype == torch.int32
    assert plan["hk"].shape[2] == max(feed.pillow_bicubic_taps(40, 24)[2].shape[1], feed.pillow_bicubic_taps(60, 24)[2].shape[1])
    for bad in [(0, 0, 41, 50), (5, 0, 5, 50), (-1, 0, 40, 50)]:
        with pytest.raises(ValueError):
            feed.crop_resize_plan([(50, 40)], [bad], 16, 24)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            feed.crop_resize([torch.zeros(8, 8, 3, dtype=torch.uint8)], [None], 4, 4)


def test_line_shards_match_reference(golden, tmp_path):
    """Rank / worker file shards, in-place epoch shuffles and repeat (dataset/dist_dataset.py:44-94): same lines in the same
    order as the reference reader, and the ranks of one world cover every file exactly once."""
    import itertools
    import types
    for name, text in golden["line_files"].items():
        (tmp_path / name).write_text(text)
    (tmp_path / "_SUCCESS").write_text("")
    assert len(golden["lines"]) == 7
    for g in golden["lines"]:
        files = sorted(str(tmp_path / n) for n in os.listdir(tmp_path))
        info = types.SimpleNamespace(id=g["worker_id"], num_workers=g["workers"]) if g["workers"] else None
        random.seed(g["seed"])
        ls = feed.LineShards(files, rank=g["rank"], world_size=g["world"], shuffle=g["shuffle"], repeat=g["repeat"],
                             worker_info=lambda info=info: info)
        assert list(itertools.islice(iter(ls), 40)) == g["lines"], g
        assert random.random() == g["next_random"]
    files = sorted(str(tmp_path / n) for n in golden["line_files"])
    for world in (2, 3, 7):
        seen = [l for r in range(world) for l in feed.LineShards(files, rank=r, world_size=world)]
        assert sorted(seen) == sorted(l for t in golden["line_files"].values() for l in t.splitlines(True))
    assert feed.split_shard(list(range(10)), 1, 3) == [3, 4, 5]
    with pytest.raises(RuntimeError):
        feed.split_shard([1], 0, 2)


def test_image_text_stream_matches_reference(golden):
    """JSON line -> sample (pretrain_dataset.py:225-262 and the image-only stream :368-394): image choice, prompt prefix,
    caption choice and MLM masking draw from `random` in the reference's order; broken lines are skipped."""
    tok = StubTokenizer("roberta")

    def probe(im):
        return torch.tensor([im.size[0], im.size[1], *im.getpixel((0, 0))])

    assert len(golden["image_text"]) == 3
    for g in golden["image_text"]:
        text = None
        if g["text"]:
            text = feed.TextPreprocessor(tok, feed.TextMasker(tok, 0.25, 4, 0.2, 3, False), max_tokens=10, max_masks=4, max_words=7,
                                         language_chosen=g["lang"])
        errors = []
        random.seed(g["seed"])
        st = feed.ImageTextStream(g["lines"], probe, text, image_key="binary", caption_key="desc", on_error=errors.append)
        samples = [[s[0].tolist()] + [None if v is None else list(v) for v in s[1:]] for s in st]
        assert samples == g["samples"], g["lang"]
        assert random.random() == g["next_random"]
        assert len(samples) >= 8 and len(errors) == (3 if g["text"] else 2)     # empty caption only matters with text
        batch = feed.collate([tuple([torch.tensor(s[0])] + s[1:]) for s in samples])
        assert batch[0].shape == (len(samples), 5) and (batch[1] is None) == (not g["text"])


def test_random_resized_crop_box_draws_what_torchvision_draws():
    """Same seed -> same crop box as transforms.RandomResizedCrop.get_params, and the same generator state afterwards (the
    fallback branch included: extreme aspect ratios never fit)."""
    tv = pytest.importorskip("torchvision.transforms")
    from PIL import Image
    n_fallback = 0
    for t, (w, h) in enumerate([(640, 480), (480, 640), (224, 224), (37, 501), (3000, 20), (20, 3000), (1, 1), (500, 333)] * 3):
        scale = [(0.2, 1.0), (0.5, 1.0), (0.9, 1.0)][t % 3]
        img = Image.new("RGB", (w, h))
        torch.manual_seed(t)
        i, j, ch, cw = tv.RandomResizedCrop.get_params(img, scale=scale, ratio=(3.0 / 4.0, 4.0 / 3.0))
        after = torch.rand(1).item()
        torch.manual_seed(t)
        box = feed.random_resized_crop_box(w, h, scale=scale)
        assert box == (j, i, j + cw, i + ch), (t, (w, h), box, (i, j, ch, cw))
        assert torch.rand(1).item() == after
        assert 0 <= box[0] < box[2] <= w and 0 <= box[1] < box[3] <= h
        n_fallback += (w, h) in [(3000, 20), (20, 3000)]
    assert n_fallback == 6
    g = torch.Generator().manual_seed(3)
    state = torch.random.get_rng_state()
    feed.random_resized_crop_box(640, 480, generator=g)
    assert torch.equal(torch.random.get_rng_state(), state)      # a private generator leaves the global one alone


def test_host_pack_gathers_bytes_with_any_thread_count():
    """xfm_host_pack (host-only entry point of the C-ABI): ragged tensors, empty segments, segment boundaries inside a thread's
    span; equal to torch.cat for 1..16 threads."""
    from xfm_b200 import lib
    g = torch.Generator().manual_seed(0)
    parts = [torch.randint(0, 256, (int(n),), dtype=torch.uint8, generator=g) for n in (0, 1, 7, 5 << 20, 3, 9 << 20, 0, 4 << 20, 11)]
    parts.append(torch.randint(0, 1000, (1000, 3), dtype=torch.int64, generator=g))
    ref = torch.cat([p.reshape(-1).view(torch.uint8) for p in parts])
    for threads in (1, 2, 3, 8, 16):
        out = torch.zeros(ref.numel() + 5, dtype=torch.uint8)
        lib.host_pack(parts, out, threads=threads)
        assert torch.equal(out[:-5], ref) and int(out[-5:].sum()) == 0
    lib.host_pack([], torch.zeros(1, dtype=torch.uint8))
    with pytest.raises(AssertionError):
        lib.host_pack([torch.zeros(4, dtype=torch.uint8)], torch.zeros(3, dtype=torch.uint8))


def test_vqa_collate_matches_reference(golden):
    g = golden["vqa_collate"][0]
    vb = [(torch.full((3, 2, 2), float(i)), f"question {i}", [f"a{i}{j}" for j in range(1 + i % 3)],
           [0.25 * (j + 1) for j in range(1 + i % 3)]) for i in range(5)]
    im, qs, ans, w, n = feed.vqa_collate(vb)
    assert im.tolist() == g["image"] and qs == g["questions"] and ans == g["answers"] and n == g["n"]
    assert w.tolist() == g["weights"] and str(w.dtype) == g["weights_dtype"] == "torch.float32"
    assert sum(n) == len(ans) == w.numel()


def test_finetune_loader_sample_logic_matches_reference(golden):
    """BASELINE configs #3 - #5: what the reference's re_train_dataset / re_eval_dataset / nlvr_dataset / vqa_dataset compute
    besides decoding pixels — the ITC `idx`, txt2img / img2txt, cleaned sentences, labels, the mirror decision and the
    answer weights — on the same annotations and `random` seed."""
    r = golden["retrieval"][0]
    index = feed.retrieval_image_index(r["train_anns"])
    assert [[k, v] for k, v in index.items()] == r["img_ids"]
    assert [[feed.pre_caption(a["caption"], 30), index[a["image_id"]]] for a in r["train_anns"]] == r["samples"]
    texts, images, txt2img, img2txt = feed.retrieval_eval_index(r["eval_anns"])
    assert texts == r["text"] and images == r["image"]
    assert [[k, v] for k, v in txt2img.items()] == r["txt2img"] and [[k, v] for k, v in img2txt.items()] == r["img2txt"]
    assert max(len(t.split(" ")) for t in texts) == 30                      # pre_caption truncates at max_words

    n = golden["nlvr"][0]
    assert [[feed.pre_caption(a["sentence"], 30), feed.nlvr_label(a)] for a in n["anns"]] == n["samples"]
    with pytest.raises(ValueError):
        feed.nlvr_label(dict(label="maybe"))

    v = golden["vqa"][0]
    for q, k, want in v["pre_question"]:
        assert feed.pre_question(q, k) == want, (q, k)
    random.seed(v["seed"])
    got = [list(feed.vqa_train_sample(a)) for a in v["anns"]]
    assert got == v["samples"]
    assert random.random() == v["next_random"]
    assert any(s[0] for s in got) and not all(s[0] for s in got)
    assert not any(s[0] for s, a in zip(got, v["anns"]) if feed.vqa_mentions_side(a["question"], a["answer"]))
    for s, a in zip(got, v["anns"]):
        assert (s[3] == [0.5]) == (a.get("dataset") == "vg") and abs(sum(s[3]) - (0.5 if a.get("dataset") == "vg" else 1.0)) < 1e-9


def test_pillow_bicubic_taps_many_axis_lengths():
    """One-row strips, 300 random (in, out) lengths from 1-pixel sources to 20x down-scaling: the tap tables evaluated in integer
    arithmetic equal PIL's horizontal BICUBIC pass everywhere (the vertical pass of a 1 -> 1 axis is the identity)."""
    np = pytest.importorskip("numpy")
    from PIL import Image
    rng = np.random.default_rng(11)
    sizes = [(1, 1), (1, 7), (2, 384), (3, 224), (4480, 224), (223, 224), (225, 224), (447, 224), (449, 224), (224, 1)]
    sizes += [(int(rng.integers(1, 2500)), int(rng.integers(1, 500))) for _ in range(290)]
    for w_in, w_out in sizes:
        strip = rng.integers(0, 256, size=(1, w_in, 3), dtype=np.uint8)
        ref = np.asarray(Image.fromarray(strip).resize((w_out, 1), Image.BICUBIC))
        first, count, taps = feed.pillow_bicubic_taps(w_in, w_out)
        assert taps.shape[1] == feed.bicubic_ksize(w_in, w_out) and int(count.max()) <= taps.shape[1]
        assert int(first.min()) >= 0 and int((first + count).max()) <= w_in
        idx = np.minimum(first[:, None].astype(np.int64) + np.arange(taps.shape[1])[None, :], w_in - 1)
        acc = (strip[0].astype(np.int64)[idx, :] * taps.astype(np.int64)[:, :, None]).sum(1) + (1 << 21)
        got = np.clip(acc >> 22, 0, 255).astype(np.uint8)
        assert (got == ref[0]).all(), (w_in, w_out)


def test_randaugment_sampling_and_table_operations_match_reference(golden):
    """dataset/randaugment.py: (1) which operations fire with which arguments — the reference's own RandomAugment.__call__ with
    its operation functions replaced by recorders — for the pre-training and the box_transform operation lists and the full
    14-operation default, same numpy.random stream afterwards; (2) Identity / AutoContrast / Equalize / Brightness outputs,
    including the reference's uint8 negation in AutoContrast."""
    np = pytest.importorskip("numpy")
    assert len(golden["randaugment"]) == 4
    seen = set()
    for g in golden["randaugment"]:
        sampler = feed.RandAugmentSampler(g["N"], g["M"], g["augs"])
        np.random.seed(g["seed"])
        for want in g["runs"]:
            got = [[n, [list(a) if isinstance(a, tuple) else a for a in args]] for n, args in sampler.sample()]
            assert got == want
            seen.update(n for n, _ in got)
        assert float(np.random.random()) == g["next_random"]
    assert seen == set(feed.RandAugmentSampler.ALL)
    private = feed.RandAugmentSampler(2, 7, ["Rotate", "ShearX"], rng=np.random.RandomState(1)).sample()
    np.random.seed(1)
    assert private == feed.RandAugmentSampler(2, 7, ["Rotate", "ShearX"]).sample()

    assert len(golden["randaugment_ops"]) == 8
    wrapped = 0
    for g in golden["randaugment_ops"]:
        img = np.array(g["image"], dtype=np.uint8)
        for key, want in g.items():
            if key == "image":
                continue
            name, _, f = key.partition(":")
            got = feed.apply_channel_tables(img, name, (float(f),) if f else ())
            assert got.dtype == np.uint8 and (got == np.array(want, dtype=np.uint8)).all(), key
        wrapped += int(img.min(axis=(0, 1)).max() > 0)
    assert wrapped >= 2                                   # channels with min > 0 exercise the wrapped offset
    with pytest.raises(ValueError):
        feed.channel_table(img[:, :, 0], "Rotate")


@pytest.mark.skipif(not os.path.isdir(os.environ.get("XFM_REFERENCE_ROOT", "")),
                    reason="XFM_REFERENCE_ROOT does not name a checkout of the original XFM sources")
def test_live_differential_against_the_reference_loader_code():
    """Beyond the committed fixture: tests/feed_probe.py imports the reference's dataset package in a subprocess and compares
    it with xfm_b200.feed on fresh random configurations and seeds (600 masker / preprocess cases over random mask
    probabilities, budgets, n-gram settings, whole-word modes and lengths; 400 boxes; 400 RandAugment draws), and runs the
    reference's four dataset classes against the classes of the same names in xfm_b200.feed on JSON-line files (every sample
    of a shuffled, rank-sharded epoch incl. the region loader's crop / flip / BICUBIC-resize pixels, and a collated batch)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "feed_probe.py"), "2026"], capture_output=True, text=True,
                       timeout=600)
    lines = [l for l in r.stdout.splitlines() if l.startswith("PROBE_JSON ")]
    assert r.returncode == 0 and lines, r.stderr[-3000:]
    res = json.loads(lines[-1][len("PROBE_JSON "):])
    assert res["mismatches"] == [], res["mismatches"]
    assert res["masker"] == 600 and res["preprocess"] == 600 and res["image_atts"] == 400 and res["randaugment"] == 400
    assert res["datasets"] >= 100      # samples of the four dataset classes compared end to end (3 rank / world settings each)


def test_text_dataset_through_a_dataloader_with_workers(tmp_path):
    """feed.TextJsonDataset under torch's DataLoader with two worker processes (the real get_worker_info): the workers split the
    rank's files, every line arrives exactly once, batches have the collate layout."""
    import json as _json
    tok = StubTokenizer("roberta")
    want = []
    for f in range(4):
        with open(tmp_path / f"part-{f}", "w") as fh:
            for j in range(3):
                text = f"the dog table {['red', 'blue', 'green'][j]} " + " ".join(["cat"] * f)
                want.append(tok.convert_tokens_to_ids([tok.cls_token] + tok.tokenize(text))[:9])
                fh.write(_json.dumps(dict(text=text)) + "\n")
    config = dict(text_encoder="roberta-base", skipgram_prb=0.2, skipgram_size=3, print_broken_data=True,
                  texts=dict(text_key="text", batch_size=4, tokenized=False, mask_prob=0.2, max_masks=3, mask_whole_word=False,
                             max_words=30, max_tokens=10))
    ds = feed.TextJsonDataset(config, str(tmp_path), rank=0, world_size=1, shuffle=False, repeat=False, tokenizer=tok)
    loader = torch.utils.data.DataLoader(ds, batch_size=ds.batch_size, num_workers=2, collate_fn=ds.collate_fn, timeout=120)
    rows = []
    for ids, atts, ids_masked, pos, mids in loader:
        assert ids.dtype == torch.int64 and ids.shape[1] == 10 and pos.shape[1] == 3 and atts.shape == ids.shape
        rows += [r[:int(a.sum()) - 1].tolist() for r, a in zip(ids, atts)]          # without the eos token
    assert sorted(rows) == sorted(want) and len(rows) == 12
    with pytest.raises(NotImplementedError):
        feed.list_files("hdfs://cluster/path")


def test_flipped_crops_reproduce_crop_hflip_resize_order():
    """crop -> hflip -> resize (region loader, pretrain_dataset.py:470-483) == resize of the mirrored crop: `flipped_crops`
    hands `crop_resize` exactly the pixels PIL's crop + transpose produce, and leaves unflagged images untouched."""
    np = pytest.importorskip("numpy")
    from PIL import Image
    from oracle.feed_oracle import pil_crop_resize
    rng = np.random.default_rng(2)
    imgs = [rng.integers(0, 256, size=(int(h), int(w), 3), dtype=np.uint8) for h, w in [(20, 30), (17, 9), (40, 40)]]
    boxes = [(3, 2, 25, 18), None, (0, 5, 40, 33)]
    tens = [torch.from_numpy(i) for i in imgs]
    out_images, out_boxes = feed.flipped_crops(tens, boxes, [1, 1, 0])
    assert out_boxes == [None, None, boxes[2]] and out_images[2] is tens[2]
    for im, bx, got in zip(imgs[:2], boxes[:2], out_images[:2]):
        pil = Image.fromarray(im)
        pil = (pil if bx is None else pil.crop(bx)).transpose(Image.FLIP_LEFT_RIGHT)
        assert got.is_contiguous() and (got.numpy() == np.asarray(pil)).all()
        assert (pil_crop_resize(got.numpy(), None, 16, 16) == np.asarray(pil.resize((16, 16), Image.BICUBIC))).all()
    assert feed.flipped_crops(tens, boxes, None) == (tens, boxes)
