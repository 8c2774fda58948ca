"""Numpy restatement of the baseline JPEG decode that `feed.decode_jpeg` runs on the GPU, and the seeded test corpus.
TEST INFRASTRUCTURE ONLY (xfm_b200/ never imports it).  Written from the algorithm, pinned to Pillow by
tests/test_jpeg_cpu.py: `decode(blob)` must equal `Image.open(BytesIO(blob)).convert("RGB")` byte for byte.

Pillow 12.2 decodes through libjpeg-turbo 3.1 (its x86-64 SIMD code), with the library defaults Pillow leaves alone:
  * Huffman decode, DC prediction reset at every restart interval, coefficients stored as int16 (JCOEF);
  * ISLOW IDCT as the SIMD code computes it: 16-bit dequantisation products and 16-bit sums where the SIMD code adds in
    16-bit lanes, 16-bit saturation of the first pass, and a final clamp to [0, 255] — not the C code's
    range_limit[x & 1023] wrap (`idct_islow`; DESIGN.md §8 records where the two differ);
  * fancy upsampling (jdsample.c h2v1 / h2v2, triangle filter with edge replication; plain replication when the
    downsampled width is <= 2);
  * jdcolor.c ycc_rgb_convert (16-bit fixed-point tables, ONE_HALF rounding, clamp)."""
import io

import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                   21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53,
                   60, 61, 54, 47, 55, 62, 63])


class Unsupported(Exception):
    """The stream is outside the device subset (it is decoded by Pillow instead)."""


def _u16(b, i):
    return (b[i] << 8) | b[i + 1]


def parse(blob):
    """Marker walk of a baseline single-scan JPEG: dict(W, H, comps [(id, h, v, tq)], qt {id: int[64] natural order},
    ht {(class, id): (counts, symbols)}, scan [(comp index, td, ta)], dri, ecs (start, end)).  Raises Unsupported."""
    b = blob
    if len(b) < 4 or b[0] != 0xFF or b[1] != 0xD8:
        raise Unsupported("no SOI")
    p, qt, ht, dri, sof, jfif, adobe = 2, {}, {}, 0, None, False, None
    while True:
        if p >= len(b) or b[p] != 0xFF:
            raise Unsupported("bytes between segments")
        while p < len(b) and b[p] == 0xFF:
            p += 1
        if p + 2 >= len(b):
            raise Unsupported("truncated")
        m = b[p]
        p += 1
        L = _u16(b, p)
        if L < 2 or p + L > len(b):
            raise Unsupported("bad length")
        seg = b[p + 2:p + L]
        if m == 0xE0 and len(seg) >= 14 and seg[:5] == b"JFIF\0":
            jfif = True
        elif m == 0xEE and len(seg) >= 12 and seg[:5] == b"Adobe":
            adobe = seg[11]
        elif m == 0xDB:
            i = 0
            while i < len(seg):
                pq, tq = seg[i] >> 4, seg[i] & 15
                if pq != 0 or tq > 3 or i + 65 > len(seg):
                    raise Unsupported("DQT")
                t = np.zeros(64, np.int64)
                t[ZIGZAG] = np.frombuffer(seg[i + 1:i + 65], np.uint8)
                qt[tq] = t
                i += 65
        elif m == 0xC4:
            i = 0
            while i < len(seg):
                tc, th = seg[i] >> 4, seg[i] & 15
                if tc > 1 or th > 1 or i + 17 > len(seg):
                    raise Unsupported("DHT")
                counts = list(seg[i + 1:i + 17])
                n = sum(counts)
                if n > 256 or i + 17 + n > len(seg):
                    raise Unsupported("DHT")
                ht[(tc, th)] = (counts, list(seg[i + 17:i + 17 + n]))
                i += 17 + n
        elif m == 0xDD:
            if len(seg) < 2:
                raise Unsupported("DRI")
            dri = _u16(seg, 0)
        elif m in (0xC0, 0xC1):
            if sof is not None or len(seg) < 6 or seg[0] != 8:
                raise Unsupported("SOF")
            H, W, nf = _u16(seg, 1), _u16(seg, 3), seg[5]
            if H == 0 or W == 0 or nf not in (1, 3) or len(seg) < 6 + 3 * nf:
                raise Unsupported("SOF")
            sof = (W, H, [(seg[6 + 3 * c], seg[7 + 3 * c] >> 4, seg[7 + 3 * c] & 15, seg[8 + 3 * c]) for c in range(nf)])
        elif m == 0xDA:
            if sof is None:
                raise Unsupported("SOS before SOF")
            W, H, comps = sof
            ns = seg[0] if seg else 0
            if ns != len(comps) or len(seg) < 4 + 2 * ns:
                raise Unsupported("scan")
            scan = []
            for c in range(ns):
                cid, t = seg[1 + 2 * c], seg[2 + 2 * c]
                if cid != comps[c][0]:
                    raise Unsupported("scan order")
                scan.append((c, t >> 4, t & 15))
            if (seg[1 + 2 * ns], seg[2 + 2 * ns], seg[3 + 2 * ns]) != (0, 63, 0):
                raise Unsupported("not sequential")
            if len(comps) == 3:
                ids = [c[0] for c in comps]
                if not jfif and ((adobe is not None and adobe == 0) or (adobe is None and ids == [82, 71, 66])):
                    raise Unsupported("RGB colour space")
            hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
            for cid, h, v, tq in comps:
                if h < 1 or v < 1 or tq not in qt or (len(comps) == 3 and (hmax // h, vmax // v) not in ((1, 1), (2, 1), (2, 2))):
                    raise Unsupported("sampling")
                if len(comps) == 3 and (hmax % h or vmax % v):
                    raise Unsupported("sampling")
            for _, td, ta in scan:
                if (0, td) not in ht or (1, ta) not in ht:
                    raise Unsupported("missing Huffman table")
            start = p + L
            q, end = start, None
            while q + 1 < len(b):
                if b[q] == 0xFF and b[q + 1] != 0x00 and not (0xD0 <= b[q + 1] <= 0xD7):
                    end = q
                    break
                q += 1
            if end is None or b[end + 1] != 0xD9:
                raise Unsupported("not a single scan ending in EOI")
            return dict(W=W, H=H, comps=comps, qt=qt, ht=ht, scan=scan, dri=dri, ecs=(start, end))
        elif m in (0xD8, 0xD9) or (0xC2 <= m <= 0xCF and m not in (0xC4, 0xC8, 0xCC)) or m == 0xCC or m == 0xDC:
            raise Unsupported(f"marker {m:02x}")
        p += L


def _huff_lut(counts, symbols):
    """16-bit window -> (symbol, code length); length 0 = invalid code."""
    sym, ln = np.zeros(65536, np.int64), np.zeros(65536, np.int64)
    code, k = 0, 0
    for l in range(1, 17):
        for _ in range(counts[l - 1]):
            lo = code << (16 - l)
            if lo + (1 << (16 - l)) > 65536:
                raise Unsupported("bad Huffman table")
            sym[lo:lo + (1 << (16 - l))], ln[lo:lo + (1 << (16 - l))] = symbols[k], l
            code += 1
            k += 1
        code <<= 1
    return sym.tolist(), ln.tolist()


def _intervals(b, start, end):
    """Split the entropy-coded segment at RST markers and remove the 0xFF00 stuffing: [(bytes, rst index or -1)]."""
    out, cur, q, rst = [], bytearray(), start, -1
    while q < end:
        c = b[q]
        if c == 0xFF:
            n = b[q + 1]
            if n == 0x00:
                cur.append(0xFF)
                q += 2
                continue
            if 0xD0 <= n <= 0xD7:
                out.append((bytes(cur), rst))
                cur, rst = bytearray(), n - 0xD0
                q += 2
                continue
            raise Unsupported("fill bytes inside the scan")
        cur.append(c)
        q += 1
    out.append((bytes(cur), rst))
    return out


def entropy_decode(info, blob):
    """Coefficients per component: int16 [bh, bw, 64] (natural order), bw x bh blocks as the scan lays them out."""
    W, H, comps = info["W"], info["H"], info["comps"]
    nc = len(comps)
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    if nc == 1:
        layout = [(0, 1, 1)]
        mx, my = -(-W // 8), -(-H // 8)
    else:
        layout = [(c, comps[c][1], comps[c][2]) for c in range(nc)]
        mx, my = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    coef = [np.zeros((my * v, mx * h, 64), np.int64) for (_, h, v) in layout]
    luts = {k: _huff_lut(*t) for k, t in info["ht"].items()}
    scan = info["scan"]
    total = mx * my
    ri = info["dri"] or total
    parts = _intervals(blob, *info["ecs"])
    if len(parts) != -(-total // ri) or any(r != (i - 1) % 8 for i, (_, r) in enumerate(parts) if i > 0):
        raise Unsupported("restart markers")
    zz = ZIGZAG.tolist()
    for iv, (data, _) in enumerate(parts):
        bits = np.unpackbits(np.frombuffer(data + b"\0\0\0", np.uint8)).astype(np.int64)
        nbits = 8 * len(data)
        win = np.zeros(nbits + 1, np.int64)
        for i in range(16):
            win += bits[i:i + nbits + 1] << (15 - i)
        win = win.tolist()
        pos = 0
        pred = [0] * nc

        def sym(tab):
            nonlocal pos
            s, l = luts[tab][0][win[pos]], luts[tab][1][win[pos]]
            if l == 0:
                raise Unsupported("invalid Huffman code")
            pos += l
            return s

        def extend(s):
            nonlocal pos
            if s == 0:
                return 0
            v = win[pos] >> (16 - s)
            pos += s
            return v if v >= (1 << (s - 1)) else v - (1 << s) + 1

        for m in range(iv * ri, min(total, (iv + 1) * ri)):
            my_, mx_ = divmod(m, mx)
            for li, (c, h, v) in enumerate(layout):
                _, td, ta = scan[c]
                for by in range(v):
                    for bx in range(h):
                        blk = coef[li][my_ * v + by, mx_ * h + bx]
                        pred[li] += extend(sym((0, td)))
                        blk[0] = ((pred[li] + 32768) & 0xFFFF) - 32768
                        k = 1
                        while k < 64:
                            rs = sym((1, ta))
                            r, s = rs >> 4, rs & 15
                            if s == 0:
                                if r != 15:
                                    break
                                if k + 15 > 63:
                                    raise Unsupported("run past coefficient 63")
                                k += 16
                                continue
                            k += r
                            if k > 63:
                                raise Unsupported("run past coefficient 63")
                            blk[zz[k]] = extend(s)
                            k += 1
            if pos > nbits:
                raise Unsupported("entropy data ends early")
    return coef


_F = dict(F029=2446, F039=3196, F054=4433, F076=6270, F089=7373, F117=9633, F150=12299, F184=15137, F196=16069,
          F205=16819, F256=20995, F307=25172)


def _s16(x):
    return ((x + 32768) & 0xFFFF) - 32768


def _dodct(x, shift):
    """One 1-D pass of the ISLOW IDCT over axis -2 of x (int64 [..., 8, n]) as the SIMD code evaluates it."""
    F = _F
    x0, x1, x2, x3, x4, x5, x6, x7 = (x[..., k, :] for k in range(8))
    tmp0, tmp1 = _s16(x0 + x4) << 13, _s16(x0 - x4) << 13
    tmp2 = x2 * F["F054"] + x6 * (F["F054"] - F["F184"])
    tmp3 = x2 * (F["F054"] + F["F076"]) + x6 * F["F054"]
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    z3, z4 = _s16(x7 + x3), _s16(x5 + x1)
    z3p = z3 * (F["F117"] - F["F196"]) + z4 * F["F117"]
    z4p = z3 * F["F117"] + z4 * (F["F117"] - F["F039"])
    o0 = x7 * (F["F029"] - F["F089"]) - x1 * F["F089"] + z3p
    o3 = -x7 * F["F089"] + x1 * (F["F150"] - F["F089"]) + z4p
    o1 = x5 * (F["F205"] - F["F256"]) - x3 * F["F256"] + z4p
    o2 = -x5 * F["F256"] + x3 * (F["F307"] - F["F256"]) + z3p
    r = 1 << (shift - 1)
    return np.stack([(t10 + o3 + r) >> shift, (t11 + o2 + r) >> shift, (t12 + o1 + r) >> shift, (t13 + o0 + r) >> shift,
                     (t13 - o0 + r) >> shift, (t12 - o1 + r) >> shift, (t11 - o2 + r) >> shift, (t10 - o3 + r) >> shift], axis=-2)


def idct_islow(coef, q):
    """coef int [..., 64] natural order, q int [64] -> uint8 [..., 8, 8]: libjpeg-turbo's jsimd_idct_islow."""
    c = coef.reshape(coef.shape[:-1] + (8, 8)).astype(np.int64)
    d = _s16(c * q.reshape(8, 8))
    ws = np.clip(_dodct(d, 11), -32768, 32767)                      # pass 1: columns (axis -2 = row index)
    dc_only = (c[..., 1:, :] == 0).all(axis=(-2, -1))               # the whole block has no vertical AC term
    ws = np.where(dc_only[..., None, None], _s16(d[..., :1, :] << 2), ws)
    out = _dodct(np.swapaxes(ws, -1, -2), 18)                        # pass 2: rows
    return (np.clip(np.swapaxes(out, -1, -2), -128, 127) + 128).astype(np.uint8)


def _upsample(p, fh, fv):
    """Plane p (downsampled size) -> libjpeg-turbo's fancy upsampling by (fh, fv) in {(1,1), (2,1), (2,2)}."""
    p = p.astype(np.int64)
    if (fh, fv) == (1, 1):
        return p
    dh, dw = p.shape
    if dw <= 2:
        return np.repeat(np.repeat(p, fh, axis=1), fv, axis=0)
    left, right = np.concatenate([p[:, :1], p[:, :-1]], 1), np.concatenate([p[:, 1:], p[:, -1:]], 1)
    out = np.empty((dh, 2 * dw), np.int64)
    if fv == 1:
        out[:, 0::2] = (3 * p + left + 1) >> 2
        out[:, 1::2] = (3 * p + right + 2) >> 2
        return out
    up, down = np.concatenate([p[:1], p[:-1]], 0), np.concatenate([p[1:], p[-1:]], 0)
    res = np.empty((2 * dh, 2 * dw), np.int64)
    for r, nb in ((0, up), (1, down)):
        cs = 3 * p + nb
        csl, csr = np.concatenate([cs[:, :1], cs[:, :-1]], 1), np.concatenate([cs[:, 1:], cs[:, -1:]], 1)
        res[r::2, 0::2] = (3 * cs + csl + 8) >> 4
        res[r::2, 1::2] = (3 * cs + csr + 7) >> 4
    return res


def ycc_to_rgb(y, cb, cr):
    x = np.arange(256, dtype=np.int64) - 128
    fix = lambda v: int(v * 65536 + 0.5)  # noqa: E731
    cr_r, cb_b = (fix(1.40200) * x + 32768) >> 16, (fix(1.77200) * x + 32768) >> 16
    cr_g, cb_g = -fix(0.71414) * x, -fix(0.34414) * x + 32768
    r = y + cr_r[cr]
    g = y + ((cb_g[cb] + cr_g[cr]) >> 16)
    b = y + cb_b[cb]
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def decode(blob):
    """uint8 [H, W, 3]: the RGB image Pillow returns for a stream of the device subset; raises Unsupported otherwise."""
    info = parse(blob)
    W, H, comps = info["W"], info["H"], info["comps"]
    coef = entropy_decode(info, blob)
    hmax, vmax = max(c[1] for c in comps), max(c[2] for c in comps)
    planes = []
    for ci, (cid, h, v, tq) in enumerate(comps):
        px = idct_islow(coef[ci], info["qt"][tq])                     # [bh, bw, 8, 8]
        bh, bw = px.shape[:2]
        plane = px.transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8)
        if len(comps) == 1:
            return np.repeat(plane[:H, :W, None], 3, axis=2)
        dw, dh = -(-W * h // hmax), -(-H * v // vmax)
        planes.append(_upsample(plane[:dh, :dw], hmax // h, vmax // v)[:H, :W])
    return ycc_to_rgb(*planes)


# ---------------------------------------------------------------------------------------------------------------- corpus
def content(rng, h, w, kind):
    """Seeded test images: smooth gradients, noise, hard edges (large IDCT overshoots at low quality)."""
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "smooth":
        img = np.stack([xx * 255 // max(w - 1, 1), yy * 255 // max(h - 1, 1), (xx + yy) * 127 // max(w + h - 2, 1)], -1)
    elif kind == "noise":
        img = rng.integers(0, 256, (h, w, 3))
    else:
        img = np.where((((xx // 3) + (yy // 5)) % 2)[..., None] == 1, [255, 0, 255], [0, 255, 0])
        img[rng.integers(0, h, max(1, h // 4)), :] = 255
    return img.astype(np.uint8)


def encode(img, gray=False, **kw):
    from PIL import Image
    pil = Image.fromarray(img)
    if gray:
        pil = pil.convert("L")
    f = io.BytesIO()
    pil.save(f, "JPEG", **kw)
    return f.getvalue()


def pil_rgb(blob):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(blob)).convert("RGB"))


def corpus(seed=0, large=True):
    """[(name, bytes)]: every width and height 1..17 and odd sizes around multiples of 8 / 16 up to 40, plus 640x480,
    481x353 and 1000x17; quality 5 .. 100, subsampling 4:4:4 / 4:2:2 / 4:2:0, optimize on / off, restart markers none /
    every block / every MCU row, grayscale; three kinds of content.  Parameters cycle / are drawn from a seeded generator
    so that every value of every axis occurs many times without the full cross product."""
    rng = np.random.default_rng(seed)
    sizes = [(w, h) for w in range(1, 18) for h in (w, 18 - w)]
    sizes += [(w, h) for w in (7, 9, 15, 17, 23, 25, 31, 33, 39) for h in (1, 9, 17, 31, 33, 40)]
    sizes += [(40, 40), (24, 16), (16, 24)]
    if large:
        sizes += [(640, 480), (481, 353), (1000, 17)]
    quals, subs, kinds = (5, 50, 75, 90, 95, 100), (0, 1, 2), ("smooth", "noise", "edges")
    rsts = ({}, {"restart_marker_blocks": 1}, {"restart_marker_rows": 1})
    out = []
    for i, (w, h) in enumerate(sizes):
        kind = kinds[i % 3]
        img = content(rng, h, w, kind)
        rst = (i // 3) % 3
        kw = dict(quality=quals[i % 6], optimize=bool(rng.integers(0, 2)), **rsts[rst])
        gray = i % 7 == 3
        if not gray:
            kw["subsampling"] = subs[(i // 2) % 3]
        name = f"{w}x{h}_{kind}_q{kw['quality']}_{'gray' if gray else 's%d' % kw['subsampling']}_o{int(kw['optimize'])}_r{rst}"
        out.append((name, encode(img, gray=gray, **kw)))
    return out
