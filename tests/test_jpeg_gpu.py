"""Baseline JPEG decode on the B200 (csrc/jpeg.cu through feed.decode_jpeg / decode_crop_resize): bit-identical to
`Image.open(f).convert("RGB")`, fallback images in place, the evaluation transform from file bytes equal to torchvision."""
import io
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import jpeg_ref as J  # noqa: E402
from test_jpeg_cpu import classified_files, overshoot_files  # noqa: E402
from xfm_b200 import feed, lib  # noqa: E402

pytestmark = pytest.mark.gpu


def _images(out, meta):
    host = out.cpu()
    return [host[o:o + w * h * 3].view(h, w, 3).numpy() for o, w, h in meta.tolist()]


def test_decode_jpeg_is_bit_identical_to_pillow_on_the_corpus():
    corpus = J.corpus(seed=0) + [(f"overshoot{i}", b) for i, b in enumerate(overshoot_files())]
    out, meta, nfb = feed.decode_jpeg([b for _, b in corpus])
    assert nfb == 0
    for (name, blob), img in zip(corpus, _images(out, meta)):
        assert np.array_equal(img, J.pil_rgb(blob)), name


def test_mixed_batch_keeps_order_and_counts_fallbacks():
    files = classified_files()
    broken = files.pop("multi_scan")[0]          # a second copy of the scan: Pillow raises on it, and so does the batch
    with pytest.raises(_pillow_outcome(broken)):
        feed.decode_jpeg([files["baseline"][0], broken])
    blobs = [b for b, _ in files.values()]
    blobs = blobs + blobs[:3]
    out, meta, nfb = feed.decode_jpeg(blobs)
    assert nfb == sum(1 for _, want in files.values() if want != 0)
    for blob, img in zip(blobs, _images(out, meta)):
        assert np.array_equal(img, J.pil_rgb(blob))


def test_restart_intervals_decode_to_the_same_bytes():
    rng = np.random.default_rng(7)
    img = J.content(rng, 97, 131, "edges")
    for sub in (0, 1, 2):
        blobs = [J.encode(img, quality=q, subsampling=sub, **kw) for q in (60, 95)
                 for kw in ({}, {"restart_marker_blocks": 1}, {"restart_marker_blocks": 3}, {"restart_marker_rows": 1})]
        out, meta, nfb = feed.decode_jpeg(blobs)
        imgs = _images(out, meta)
        assert nfb == 0
        for k in range(4):
            assert np.array_equal(imgs[k], imgs[0]) and np.array_equal(imgs[4 + k], imgs[4])
            assert np.array_equal(imgs[k], J.pil_rgb(blobs[k]))


@pytest.mark.parametrize("res", [224, 384, 480])
def test_evaluation_transform_from_file_bytes_equals_torchvision(res):
    from PIL import Image
    from torchvision import transforms
    rng = np.random.default_rng(res)
    blobs = [J.encode(J.content(rng, h, w, k), quality=90, subsampling=s)
             for (w, h), k, s in zip([(640, 480), (481, 353), (300, 500), (97, 61)], ("noise", "smooth", "edges", "noise"), (2, 1, 0, 2))]
    tf = transforms.Compose([transforms.Resize((res, res), interpolation=transforms.InterpolationMode.BICUBIC),
                             transforms.ToTensor(), transforms.Normalize(feed.CLIP_MEAN, feed.CLIP_STD)])
    want = torch.stack([tf(Image.open(io.BytesIO(b)).convert("RGB")) for b in blobs])
    got = lib.image_u8_to_f32(feed.decode_crop_resize(blobs, [None] * len(blobs), res, res), feed.CLIP_MEAN, feed.CLIP_STD)
    assert torch.equal(got.cpu(), want)
    g = torch.Generator().manual_seed(res)
    boxes = [feed.random_resized_crop_box(*feed.jpeg_size(b), generator=g) for b in blobs]
    got = feed.decode_crop_resize(blobs, boxes, res, res).cpu().numpy()
    for b, bx, img in zip(blobs, boxes, got):
        want = np.asarray(Image.open(io.BytesIO(b)).convert("RGB").crop(bx).resize((res, res), Image.BICUBIC))
        assert np.array_equal(img, want)


def test_output_bytes_outside_the_images_are_untouched():
    """Call the C-ABI directly with gaps of canary bytes between, before and after the images."""
    rng = np.random.default_rng(9)
    blobs = [J.encode(J.content(rng, h, w, "noise"), quality=80, subsampling=s, **kw)
             for (w, h), s, kw in [((17, 9), 2, {}), ((33, 40), 1, {"restart_marker_blocks": 1}), ((8, 8), 0, {})]]
    blobs.insert(1, J.encode(J.content(rng, 5, 7, "noise"), quality=80, progressive=True))     # fallback: not touched
    info = lib.jpeg_plan(blobs)
    gap = 37
    offs = np.zeros((len(blobs), 4), np.int64)
    dev = info[:, 0] == 0
    lens = np.array([len(b) for b in blobs])
    offs[:, 0] = np.cumsum(np.where(dev, lens, 0)) - np.where(dev, lens, 0)
    offs[:, 1] = np.cumsum(np.where(dev, info[:, 4], 0)) - np.where(dev, info[:, 4], 0)
    offs[:, 2] = np.cumsum(np.where(dev, info[:, 5], 0)) - np.where(dev, info[:, 5], 0)
    sizes = info[:, 1] * info[:, 2] * 3
    offs[:, 3] = np.cumsum(sizes + gap) - sizes
    desc, iv = lib.jpeg_tables(blobs, info, offs)
    data = torch.frombuffer(bytearray(b"".join(b for b, d in zip(blobs, dev) if d)), dtype=torch.uint8).cuda()
    out = torch.full((int(offs[-1, 3] + sizes[-1] + gap),), 0xA5, dtype=torch.uint8, device="cuda")
    coef = torch.empty((int(info[dev, 4].sum()), 64), dtype=torch.int16, device="cuda")
    planes = torch.empty(int(info[dev, 5].sum()), dtype=torch.uint8, device="cuda")
    status = torch.from_numpy(np.where(dev, 0, 1).astype(np.int32)).cuda()
    lib.jpeg_decode(data, desc.cuda(), iv.cuda(), len(blobs), coef, planes, out, status, int(info[dev, 4].max()),
                    int(info[dev, 1].max()), int(info[dev, 2].max()))
    host = out.cpu().numpy()
    mask = np.ones(host.size, bool)
    for i, b in enumerate(blobs):
        if dev[i]:
            mask[offs[i, 3]:offs[i, 3] + sizes[i]] = False
            assert np.array_equal(host[offs[i, 3]:offs[i, 3] + sizes[i]].reshape(info[i, 2], info[i, 1], 3), J.pil_rgb(b))
    assert (host[mask] == 0xA5).all()
    assert status.cpu().tolist() == [0, 1, 0, 0]


def _pillow_outcome(blob):
    try:
        return J.pil_rgb(blob)
    except Exception as e:      # noqa: BLE001 — the type is what is compared
        return type(e)


def test_corrupted_and_truncated_files_give_what_pillow_gives():
    rng = np.random.default_rng(11)
    base = [J.encode(J.content(rng, 40, 56, "noise"), quality=90, subsampling=2),
            J.encode(J.content(rng, 40, 56, "smooth"), quality=75, subsampling=0, restart_marker_blocks=2)]
    cases = []
    for blob in base:
        sos = blob.index(b"\xff\xda")
        for k in range(12):
            b = bytearray(blob)
            pos = int(rng.integers(sos + 14, len(b) - 2))
            b[pos] ^= int(rng.integers(1, 256))
            cases.append(bytes(b))
        cases += [blob[:n] for n in (len(blob) - 1, len(blob) - 2, len(blob) // 2, sos + 20)]
    for blob in cases:
        want = _pillow_outcome(blob)
        if isinstance(want, type):
            with pytest.raises(want):
                feed.decode_jpeg([blob])
        else:
            out, meta, _ = feed.decode_jpeg([blob])
            assert np.array_equal(_images(out, meta)[0], want)


def test_empty_and_single_batches_and_three_kernels_per_call():
    out, meta, nfb = feed.decode_jpeg([])
    assert meta.shape == (0, 3) and nfb == 0
    assert feed.decode_crop_resize([], [], 32, 32).shape == (0, 32, 32, 3)
    blob = J.encode(J.content(np.random.default_rng(12), 30, 50, "edges"), quality=85)
    out, meta, nfb = feed.decode_jpeg([blob])
    assert np.array_equal(_images(out, meta)[0], J.pil_rgb(blob)) and nfb == 0
    blobs = [blob, J.encode(J.content(np.random.default_rng(13), 64, 64, "noise"), quality=70, restart_marker_rows=1)]
    feed.decode_jpeg(blobs)
    torch.cuda.synchronize()
    n0 = lib.launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        feed.decode_jpeg(blobs)
        torch.cuda.synchronize()
    assert lib.launch_count() - n0 == 3
    names = sorted(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "jpeg_" in e.name)
    assert len(names) == 3 and all(any(k in n for n in names) for k in ("jpeg_entropy", "jpeg_idct", "jpeg_color")), names
