"""xfm_attention_varlen_fwd / _bwd (csrc/attention_vtc.cu) against the fp64 reference and per-element bounds of
test_attention_paths_gpu.py, sequence by sequence, for packed batches of 1..128-token sequences.

Every output lives in a canary-filled buffer (dq / dk / dv as column slices of one wider buffer, as in the model); the
dropout mask is recovered bit for bit with probe inputs (q = 0, one-hot V or dO rows) and compared with
oracle/dropout_mask over the PADDED numbering attention_index(n, H, Lpad, Lpad); with dropout on, the packed outputs of the
real rows are compared with the mma.sync kernels run on the padded layout with a key mask.
"""
import ctypes as C
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from canary import Buf  # noqa: E402
from test_attention_paths_gpu import C_GRAD, C_LSE, C_OUT, SCALE, U_BF16, Case, _ratio, reference  # noqa: E402

from oracle import dropout_mask as DM  # noqa: E402

pytestmark = pytest.mark.gpu
F32, BF16 = torch.float32, torch.bfloat16
H = 12
CONST = dict(out=C_OUT, lse=C_LSE, dq=C_GRAD, dk=C_GRAD, dv=C_GRAD)
KERNELS = {"vattn_fwd_tc_kernel", "vattn_bwd_tc_kernel", "attn_delta_kernel"}


@pytest.fixture(scope="module")
def lib():
    from xfm_b200 import lib as L

    L.lib()
    L.seed_salt_set(0)   # the dropout masks below depend on dropout_seed only
    return L


def lengths_of(kind):
    if kind == "all1":
        return [1] * 300
    if kind == "all128":
        return [128] * 40
    if kind == "all40":
        return [40] * 120
    rng = np.random.default_rng(7)
    return rng.integers(1, 129, 420).tolist()   # about 200 tiles: more than one per SM


def kernel_names(fn, repeat=3):
    """Names of the CUDA kernels fn() launches, over `repeat` calls (a profiler session late in a long test run can miss a
    few kernel events; every kernel of fn() shows up in at least one of the calls)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        for _ in range(repeat):
            fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def attn_names(names):
    out = set()
    for n in names:
        m = re.search(r"\b(\w*attn\w*_kernel)\b", n)
        if m:
            out.add(m.group(1))
    return out


class Packed:
    """Inputs and canary-guarded outputs of one packed batch."""

    def __init__(self, lengths, Lpad, seed, q_zero=False):
        g = torch.Generator(device="cuda").manual_seed(seed)
        self.lengths, self.Lpad = list(lengths), Lpad
        self.n = len(lengths)
        self.T = T = int(sum(lengths))
        W = H * 64
        self.qkv = torch.randn((T, 3 * W), generator=g, device="cuda").to(BF16)
        if q_zero:
            self.qkv[:, :W] = 0
        self.q, self.k, self.v = self.qkv[:, :W], self.qkv[:, W:2 * W], self.qkv[:, 2 * W:]
        self.dout = torch.randn((T, W), generator=g, device="cuda").to(BF16)
        self.out = Buf(T, W, W + 8, BF16, off=5 * 8)
        self.lse = Buf(H, T, T, F32, off=3)
        self.delta = Buf(H, T, T, F32, off=1)
        self.grad = Buf(T, 3 * W, 3 * W + 16, BF16, off=8)
        gv = self.grad.view
        self.dq, self.dk, self.dv = gv[:, :W], gv[:, W:2 * W], gv[:, 2 * W:]
        from xfm_b200 import lib as L
        cu, tiles = L.varlen_plan(lengths)
        self.cu_host = cu
        self.cu, self.tiles = cu.cuda(), tiles.cuda()
        self.n_tiles = tiles.numel() - 1
        for b in (self.out, self.lse, self.delta, self.grad):
            b.snapshot()

    def params(self, L, p, seed):
        P = L.VarlenParams()
        P.q, P.k, P.v = self.q.data_ptr(), self.k.data_ptr(), self.v.data_ptr()
        P.q_stride = P.k_stride = P.v_stride = self.qkv.stride(0)
        P.out, P.o_stride, P.lse = self.out.view.data_ptr(), self.out.view.stride(0), self.lse.view.data_ptr()
        P.cu_seqlens, P.tiles = self.cu.data_ptr(), self.tiles.data_ptr()
        P.n, P.n_tiles, P.H, P.Lpad, P.T = self.n, self.n_tiles, H, self.Lpad, self.T
        P.scale, P.dropout_p, P.dropout_seed = SCALE, p, seed
        P.dout, P.do_stride, P.delta = self.dout.data_ptr(), self.dout.stride(0), self.delta.view.data_ptr()
        P.dq, P.dk, P.dv = self.dq.data_ptr(), self.dk.data_ptr(), self.dv.data_ptr()
        P.dq_stride = P.dk_stride = P.dv_stride = self.grad.view.stride(0)
        return P

    def run(self, L, p, seed, bwd=True):
        P = self.params(L, p, seed)
        L.check(L.lib().xfm_attention_varlen_fwd(C.byref(P), L.stream_ptr()), "xfm_attention_varlen_fwd")
        if bwd:
            L.check(L.lib().xfm_attention_varlen_bwd(C.byref(P), L.stream_ptr()), "xfm_attention_varlen_bwd")

    def groups(self):
        """{length: [sequence indices]}"""
        gs = {}
        for s, l in enumerate(self.lengths):
            gs.setdefault(l, []).append(s)
        return gs

    def rows(self, seqs, l):
        cu = self.cu_host
        return torch.cat([torch.arange(int(cu[s]), int(cu[s]) + l) for s in seqs]).cuda()


def padded_index(seqs, l, Lpad):
    """[len(seqs), H, l, l] of DM.attention_index(n, H, Lpad, Lpad)[seqs, :, :l, :l], without the whole array."""
    lke = (Lpad + 1) & ~1
    s = np.asarray(seqs, dtype=np.uint64).reshape(-1, 1, 1, 1)
    h = np.arange(H, dtype=np.uint64).reshape(1, -1, 1, 1)
    i = np.arange(l, dtype=np.uint64).reshape(1, 1, -1, 1)
    j = np.arange(l, dtype=np.uint64).reshape(1, 1, 1, -1)
    return ((s * np.uint64(H) + h) * np.uint64(Lpad) + i) * np.uint64(lke) + j


def keep_packed(seqs, l, Lpad, p, seed):
    """[len(seqs), H, l, l] kept set of sequences `seqs` under the padded numbering."""
    return torch.from_numpy(DM.keep(seed, padded_index(seqs, l, Lpad), p)).cuda()


def _heads(x, n, l):
    return x.double().reshape(n, l, H, 64).permute(0, 2, 1, 3)


def check_against_reference(pk, p, seed, record, tag):
    worst = {}
    for l, seqs in sorted(pk.groups().items()):
        rows = pk.rows(seqs, l)
        n = len(seqs)
        t = dict(q=pk.q[rows], k=pk.k[rows], v=pk.v[rows], dout=pk.dout[rows], out=types.SimpleNamespace(view=pk.out.view[rows]),
                 Bkv=n, kv_index=None)
        c = Case(id="varlen", kernels=(), B=n, H=H, Lq=l, Lk=l, drop=p)
        keep = keep_packed(seqs, l, pk.Lpad, p, seed) if p else None
        r, m = reference(c, t, keep)
        g = dict(out=_heads(pk.out.view[rows], n, l), lse=pk.lse.view[:, rows].double().view(H, n, l).permute(1, 0, 2),
                 dq=_heads(pk.dq[rows], n, l), dk=_heads(pk.dk[rows], n, l), dv=_heads(pk.dv[rows], n, l))
        for name, val in g.items():
            assert torch.isfinite(val).all(), (name, l)
            err = (val - r[name]).abs()
            rest = U_BF16 * r[name].abs() if name != "lse" else 0.0
            worst[name] = max(worst.get(name, 0.0), float(_ratio(err, CONST[name] * m[name] + rest).max()))
        dl = pk.delta.view[:, rows].double().view(H, n, l).permute(1, 0, 2)
        worst["delta"] = max(worst.get("delta", 0.0), float(_ratio((dl - r["delta"]).abs(), 2.0 ** -17 * m["delta"]).max()))
    record("varlen_case", case=tag, worst_ratio=worst)
    print(tag, worst)
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad


@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("kind", ["all1", "all128", "all40", "random"])
def test_varlen_case(lib, record, kind, p):
    lengths = lengths_of(kind)
    seed = 11 + len(lengths)
    pk = Packed(lengths, 128, seed)
    names = attn_names(kernel_names(lambda: pk.run(lib, p, seed)))
    assert names == KERNELS, names
    for b in (pk.out, pk.lse, pk.delta):
        assert b.outside_unchanged(), "written outside the view"
    assert pk.grad.outside_unchanged([pk.dq, pk.dk, pk.dv]), "dq / dk / dv written outside their column slices"
    check_against_reference(pk, p, seed, record, "%s p=%g" % (kind, p))


def test_backward_is_deterministic(lib):
    pk = Packed(lengths_of("random"), 128, 5)
    pk.run(lib, 0.1, 9)
    first = pk.grad.view.clone()
    pk.run(lib, 0.1, 9)
    assert torch.equal(first, pk.grad.view)


@pytest.mark.parametrize("Lpad", [128, 131])
def test_dropout_mask_is_the_padded_hash(lib, Lpad):
    """q = 0 makes every probability 1 / len; a one-hot V row (key j -> column j mod 64) puts P~[i, j] into out[i, j mod 64],
    a one-hot dO row (query i -> column i mod 64) puts P~[i, j] into dV[j, i mod 64]: non-zero exactly when kept."""
    p, seed = 0.3, 77
    rng = np.random.default_rng(3)
    lengths = rng.integers(1, 129, 150).tolist() + [128, 1, 64, 65]
    pk = Packed(lengths, Lpad, 21, q_zero=True)
    W = H * 64
    pos = torch.cat([torch.arange(l) for l in lengths]).cuda()          # position of every packed row in its sequence
    fwd_kept, bwd_kept = {}, {}
    for half in (0, 1):
        sel = (pos // 64 == half)
        onehot = torch.zeros((pk.T, 64), device="cuda")
        onehot[sel, pos[sel] % 64] = 1.0
        pk.qkv[:, 2 * W:] = onehot.repeat(1, H).to(BF16)
        pk.dout.copy_(onehot.repeat(1, H).to(BF16))
        pk.run(lib, p, seed)
        o = pk.out.view.float().view(pk.T, H, 64)
        dv = pk.dv.float().view(pk.T, H, 64)
        for l, seqs in pk.groups().items():
            rows = pk.rows(seqs, l)
            n = len(seqs)
            # out[i, h, c]: key 64 * half + c of query i;  dv[j, h, c]: query 64 * half + c of key j
            fo = o[rows].view(n, l, H, 64).permute(0, 2, 1, 3) != 0           # [n, H, i, c]
            fb = dv[rows].view(n, l, H, 64).permute(0, 2, 3, 1) != 0          # [n, H, c, j]
            w = min(64, l - 64 * half)
            if w <= 0:
                continue
            fwd_kept.setdefault(l, torch.zeros((n, H, l, l), dtype=torch.bool, device="cuda"))[..., 64 * half:64 * half + w] = fo[..., :w]
            bwd_kept.setdefault(l, torch.zeros((n, H, l, l), dtype=torch.bool, device="cuda"))[:, :, 64 * half:64 * half + w, :] = fb[:, :, :w, :]
    n_checked = 0
    for l, seqs in pk.groups().items():
        want = keep_packed(seqs, l, Lpad, p, seed)
        assert torch.equal(fwd_kept[l], want), ("forward mask", l)
        assert torch.equal(bwd_kept[l], want), ("backward mask", l)
        n_checked += want.numel()
    assert n_checked > 10 ** 6
    full = DM.attention_index(8, H, Lpad, Lpad)   # padded_index is the oracle's numbering
    for s in range(8):
        assert np.array_equal(padded_index([s], lengths[s], Lpad)[0], full[s, :, :lengths[s], :lengths[s]])


def test_dropout_agrees_with_padded_mma_sync(lib, record):
    """With dropout on, the packed forward / backward of the real rows match the mma.sync kernels on the padded layout with
    an additive key mask (same seed, same numbering)."""
    p, seed = 0.1, 123
    rng = np.random.default_rng(11)
    Lpad = 96
    lengths = rng.integers(1, Lpad + 1, 64).tolist()
    pk = Packed(lengths, Lpad, 31)
    pk.run(lib, p, seed)
    n, W = pk.n, H * 64
    real = torch.cat([torch.arange(s * Lpad, s * Lpad + l) for s, l in enumerate(lengths)]).cuda()
    qkv = torch.zeros((n * Lpad, 3 * W), dtype=BF16, device="cuda")
    qkv[real] = pk.qkv
    dout = torch.zeros((n * Lpad, W), dtype=BF16, device="cuda")
    dout[real] = pk.dout
    kmask = torch.full((n, Lpad), -10000.0, device="cuda")
    kmask.view(-1)[real] = 0.0
    q, k, v = qkv[:, :W], qkv[:, W:2 * W], qkv[:, 2 * W:]
    out, lse = lib.attention_fwd(q, k, v, n, H, Lpad, Lpad, SCALE, kmask=kmask, dropout_p=p, dropout_seed=seed, allow_tc=False)
    dqkv = torch.empty_like(qkv)
    lib.attention_bwd(dout, q, k, v, out, lse, n, H, Lpad, Lpad, SCALE, dqkv[:, :W], dqkv[:, W:2 * W], dqkv[:, 2 * W:],
                      kmask=kmask, dropout_p=p, dropout_seed=seed, allow_tc=False)
    mine = dict(out=pk.out.view, dq=pk.dq, dk=pk.dk, dv=pk.dv)
    theirs = dict(out=out[real], dq=dqkv[real, :W], dk=dqkv[real, W:2 * W], dv=dqkv[real, 2 * W:])
    rel = {}
    for name in mine:
        a, b = mine[name].float(), theirs[name].float()
        scale = float(b.abs().max())
        rel[name] = float((a - b).abs().max()) / scale
    lse_err = float((pk.lse.view - lse.view(n, H, Lpad).permute(1, 0, 2).reshape(H, -1)[:, real]).abs().max())
    record("varlen_vs_mma_sync", rel=rel, lse_abs=lse_err)
    print("packed vs padded mma.sync", rel, "lse", lse_err)
    # two bf16 results of the same products in a different summation order; a wrong mask would differ by O(1)
    assert all(v < 2e-2 for v in rel.values()), rel
    assert lse_err < 1e-4


def test_rejects_bad_arguments(lib):
    pk = Packed([5, 7], 8, 1)
    P = pk.params(lib, 0.0, 0)
    P.q_stride = 3 * H * 64 + 4
    assert lib.lib().xfm_attention_varlen_fwd(C.byref(P), lib.stream_ptr()) == -2
    P = pk.params(lib, 0.0, 0)
    P.q = pk.q.data_ptr() + 2
    assert lib.lib().xfm_attention_varlen_fwd(C.byref(P), lib.stream_ptr()) == -2
    P = pk.params(lib, 0.0, 0)
    P.dq = 0
    assert lib.lib().xfm_attention_varlen_bwd(C.byref(P), lib.stream_ptr()) == -2
    assert "varlen" in lib.lib().xfm_last_error().decode()
