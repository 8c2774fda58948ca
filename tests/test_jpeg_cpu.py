"""Baseline JPEG decode, CPU side: the numpy restatement (tests/jpeg_ref.py) equals Pillow byte for byte on a seeded corpus,
and the host marker walk (`xfm_jpeg_plan` / `xfm_jpeg_tables`, C++) classifies files and survives hostile input."""
import io
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import jpeg_ref as J  # noqa: E402
from xfm_b200 import lib  # noqa: E402


def _built():
    return os.path.exists(lib.LIB_PATH)


@pytest.mark.parametrize("name,blob", J.corpus(seed=0), ids=lambda v: v if isinstance(v, str) else "")
def test_numpy_restatement_equals_pillow(name, blob):
    assert np.array_equal(J.decode(blob), J.pil_rgb(blob)), name


def _patch_dqt(blob, value_dc, value_ac):
    """Rewrite every quantisation table of a quality-100 file: the same entropy data now dequantises to values far outside
    [0, 255] — Pillow's libjpeg-turbo clamps where its C IDCT would wrap through range_limit[x & 1023]."""
    b, p = bytearray(blob), 2
    while b[p + 1] != 0xDA:
        L = (b[p + 2] << 8) | b[p + 3]
        if b[p + 1] == 0xDB:
            for i in range(p + 4, p + 2 + L, 65):
                for k in range(64):
                    b[i + 1 + k] = value_dc if k < 10 else value_ac
        p += 2 + L
    return bytes(b)


def overshoot_files(seed=1):
    rng = np.random.default_rng(seed)
    return [_patch_dqt(J.encode(J.content(rng, 40, 56, kind), quality=100, subsampling=sub), 255, 97)
            for kind in ("edges", "noise") for sub in (0, 2)]


def test_numpy_restatement_equals_pillow_on_idct_overshoots():
    for blob in overshoot_files():
        assert np.array_equal(J.decode(blob), J.pil_rgb(blob))


def exif_thumbnail_file():
    """A JPEG whose APP1 segment carries a complete JPEG thumbnail (its own SOI ... EOI), as cameras write them."""
    rng = np.random.default_rng(3)
    thumb = J.encode(J.content(rng, 16, 16, "noise"), quality=80)
    main = J.encode(J.content(rng, 48, 64, "smooth"), quality=85)
    app1 = b"Exif\0\0" + b"II*\0\x08\0\0\0" + thumb
    return main[:2] + b"\xff\xe1" + (len(app1) + 2).to_bytes(2, "big") + app1 + main[2:]


def classified_files():
    from PIL import Image
    rng = np.random.default_rng(2)
    img = J.content(rng, 33, 47, "noise")
    f = io.BytesIO()
    Image.fromarray(img).save(f, "PNG")
    cmyk = io.BytesIO()
    Image.fromarray(img).convert("CMYK").save(cmyk, "JPEG", quality=90)
    # 4:4:0 (h1v2 chroma): rewrite the luma sampling byte of a 4:4:4 file from 0x11 to 0x12
    b444 = bytearray(J.encode(img, quality=90, subsampling=0))
    i = b444.index(b"\xff\xc0")
    b444[i + 11] = 0x12
    # a second scan: a progressive file is multi-scan; a baseline file with two SOS segments is the other case
    base = J.encode(img, quality=90, subsampling=2)
    eoi = base.rindex(b"\xff\xd9")
    sos = base.index(b"\xff\xda")
    two_scans = base[:eoi] + base[sos:]
    return {
        "baseline": (J.encode(img, quality=90), 0),
        "gray": (J.encode(img, gray=True, quality=90), 0),
        "exif_thumbnail": (exif_thumbnail_file(), 0),
        "progressive": (J.encode(img, quality=90, progressive=True), 3),
        "cmyk": (cmyk.getvalue(), 4),
        "h1v2": (bytes(b444), 5),
        "multi_scan": (two_scans, 7),
        "png": (f.getvalue(), 1),
    }


@pytest.mark.skipif(not _built(), reason="libxfm_b200.so not built")
def test_host_plan_classifies_files():
    files = classified_files()
    info = lib.jpeg_plan([b for b, _ in files.values()], threads=3)
    for (name, (blob, want)), row in zip(files.items(), info):
        assert int(row[0]) == want, (name, row)
        if want == 0:
            h, w = J.pil_rgb(blob).shape[:2]
            assert (int(row[1]), int(row[2])) == (w, h), name
    # the restatement agrees on what it decodes
    for name in ("baseline", "gray", "exif_thumbnail"):
        blob = files[name][0]
        assert np.array_equal(J.decode(blob), J.pil_rgb(blob)), name


@pytest.mark.skipif(not _built(), reason="libxfm_b200.so not built")
def test_host_plan_geometry_and_restart_intervals():
    rng = np.random.default_rng(4)
    img = J.content(rng, 37, 53, "edges")
    blobs = [J.encode(img, quality=75, subsampling=2), J.encode(img, quality=75, subsampling=2, restart_marker_blocks=1),
             J.encode(img, quality=75, subsampling=1, restart_marker_rows=1), J.encode(img, gray=True, quality=75)]
    info = lib.jpeg_plan(blobs)
    assert info[:, 0].tolist() == [0, 0, 0, 0]
    # 4:2:0: MCUs of 16 x 16 -> 4 x 3; blocks = 4 * 12 (Y) + 2 * 12 (Cb, Cr)
    assert info[0, 3] == 1 and info[0, 4] == 72 and info[0, 5] == 72 * 64
    assert info[1, 3] == 12
    assert info[2, 3] == 5 and info[2, 4] == 4 * 5 * 4           # 4:2:2: MCUs 16 x 8 -> 4 x 5, 4 blocks each
    assert info[3, 3] == 1 and info[3, 4] == 7 * 5
    offs = np.zeros((4, 4), np.int64)
    offs[:, 0] = np.cumsum([len(b) for b in blobs]) - [len(b) for b in blobs]
    desc, iv = lib.jpeg_tables(blobs, info, offs)
    assert iv.shape == (1 + 12 + 5 + 1, 2)
    iv = iv.numpy()
    assert (iv[:, 0] <= iv[:, 1]).all() and (np.diff(iv[:, 0]) > 0).all()
    joined = b"".join(blobs)
    for k in range(1, 12):                                     # interval k of image 1 starts right after RST(k-1)
        assert joined[iv[1 + k, 0] - 2:iv[1 + k, 0]] == bytes([0xFF, 0xD0 + (k - 1) % 8])
    assert joined[iv[12, 1]:iv[12, 1] + 2] == b"\xff\xd9"


@pytest.mark.skipif(not _built(), reason="libxfm_b200.so not built")
def test_host_plan_survives_truncation_and_corrupted_segments():
    """Every truncation of a small file, and every single-byte change inside its marker segments: the parser returns fallback
    or a consistent plan, and reads nothing outside the blob (each blob is copied into an exactly sized buffer)."""
    rng = np.random.default_rng(5)
    blob = J.encode(J.content(rng, 9, 11, "noise"), quality=50, subsampling=2, restart_marker_blocks=1)
    sos = blob.index(b"\xff\xda")
    hdr_end = sos + 2 + ((blob[sos + 2] << 8) | blob[sos + 3])
    cases = [blob[:n] for n in range(len(blob))]
    for pos in range(2, hdr_end):
        for v in (0x00, 0xFF, blob[pos] ^ 0x01, blob[pos] ^ 0x80):
            b = bytearray(blob)
            b[pos] = v
            cases.append(bytes(b))
    info = lib.jpeg_plan(cases, threads=4)
    for b, row in zip(cases, info):
        if row[0] != 0:
            continue
        assert len(b) == len(blob) and row[1] > 0 and row[2] > 0 and row[3] >= 1
        offs = np.zeros((1, 4), np.int64)
        _, iv = lib.jpeg_tables([b], row[None], offs)
        assert (iv.numpy()[:, 0] >= 0).all() and (iv.numpy()[:, 1] <= len(b)).all()
    assert (info[:len(blob), 0] != 0).all()                   # every truncation falls back
    assert info[len(blob):, 0].tolist().count(0) > 0            # some header edits stay decodable (e.g. APP0 contents)
