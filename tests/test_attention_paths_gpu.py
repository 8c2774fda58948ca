"""xfm_attention_fwd / xfm_attention_bwd against an fp64 reference of the same operation, kernel path by kernel path.

Every row of CASES is chosen to reach the kernel instantiations it names (worked out from attention.cu's attention_fwd /
attention_bwd and the *_supported() functions of attention_tc.cu, attention_xtc.cu and attention_stc.cu); the profiler
checks each row, and test_every_instantiation_is_reached checks that the rows together run every instantiation the
dispatch can choose.  The reference is plain torch in float64 on the same bf16 operands, with the dropout mask of
oracle/dropout_mask.py.  Errors are bounded per element by a magnitude tensor of the same shape (C_OUT .. C_DS below), never
relative to the largest value of the tensor, so a wrong row of a small head or of an image with one sample cannot hide
behind a large one elsewhere.  out, lse, delta, dq, dk, dv and the dS dump live inside canary-filled buffers, dq / dk / dv
as the column slices of one wider buffer that the model uses, and every byte outside the views must survive the call.

The dropout mask of each kernel is recovered bit for bit with probe inputs (test_dropout_mask_is_the_hash): q = 0 makes
every probability 1 / Lk, and one-hot rows of V (forward), dO (dV) or K (dQ) on a 64-wide window put the probability of
one (query, key) pair into one output element, which is non-zero exactly when that pair is kept.
"""
import ctypes as C
import math
import os
import re
import sys
from dataclasses import dataclass

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from canary import Buf  # noqa: E402

from oracle import dropout_mask as DM  # noqa: E402

pytestmark = pytest.mark.gpu

# Per-element error bounds: |got - ref| <= C * magnitude + 2^-8 * (|ref| + n_round * magnitude), n_round counting the bf16
# roundings of partial sums (dQ reduce-added across key-block launches, dK / dV across sample chunks of one image).
# Each C is the smallest power of two that every row of CASES passes on a B200 (NVIDIA B200, 1000 W power limit).
C_OUT = 2.0 ** -6    # out:  |P~| . |V|
C_LSE = 2.0 ** -18   # lse:  sum_j P_ij (|s_ij| + |addend_ij|) + 1
C_GRAD = 2.0 ** -6   # dq:   scale (P o (|dO| |V|^T / (1-p) + |delta|)) . |K|,  dk likewise with |Q|,  dv: |P~|^T . |dO|
C_DS = 2.0 ** -6     # dS dump: P o (|dO| |V|^T / (1-p) + |delta|)
U_BF16 = 2.0 ** -8
SCALE = 0.125
F32, BF16 = torch.float32, torch.bfloat16


@pytest.fixture(scope="module")
def lib():
    from xfm_b200 import lib as L

    L.lib()
    L.seed_salt_set(0)   # the dropout masks below depend on dropout_seed only
    return L


def _r8(x):
    return (x + 7) // 8 * 8


# ------------------------------------------------------------------------------------------------ kernel names
def _nb(L):   # internal.h KeyBlocks::nb
    return 1 if L <= 208 else (L // 192 if L % 192 <= 16 else L // 192 + 1)


def mma(fwd, dq, dkv):
    """The mma.sync family: (WARPS, STREAM) of each of the three kernels."""
    f = lambda n, w: "%s<%d,%s>" % (n, w[0], "true" if w[1] else "false")
    return (f("attn_fwd_kernel", fwd), "attn_delta_kernel", f("attn_bwd_dq_kernel", dq), f("attn_bwd_dkv_kernel", dkv))


def vit(W, table):
    nb = _nb(W * W + 1)
    names = ["vit_attn_fwd_tc_kernel<%d,%d,%s>" % (W, kb, "true" if table else "false") for kb in range(nb)]
    names += ["vit_attn_bwd_fused_tc_kernel<%d,%d,false>" % (W, kb) for kb in range(nb)]
    return tuple(names) + (("merge_parts_kernel<%d>" % nb,) if nb > 1 else ()) + ("attn_delta_kernel",)


def xtc(Lk):
    nb = _nb(Lk)
    names = ["xattn_fwd_tc_kernel<40,%d,6,%d>" % (Lk, kb) for kb in range(nb)]
    names += ["xattn_bwd_fused_tc_kernel<40,%d,%d>" % (Lk, kb) for kb in range(nb)]
    return tuple(names) + (("merge_parts_kernel<%d>" % nb,) if nb > 1 else ()) + ("attn_delta_kernel",)


STC = ("sattn_fwd_tc_kernel", "sattn_bwd_tc_kernel", "attn_delta_kernel")

# Every attention instantiation attention_fwd / attention_bwd can launch.  attn_bwd_dkv_kernel<4, true> needs at most
# 256 keys with queries that do not fit shared memory (Lq >~ 770); the other mma.sync variants follow from Lq / Lk > 256 and
# RESIDENT_SMEM_MAX.
REACHABLE = set()
for _k in ("attn_fwd_kernel", "attn_bwd_dq_kernel", "attn_bwd_dkv_kernel"):
    REACHABLE |= {"%s<%d,%s>" % (_k, w, s) for w in (4, 8) for s in ("false", "true")}
for _W in (4, 7, 12, 14, 24, 30):
    REACHABLE |= set(vit(_W, True)) | set(vit(_W, False))
for _Lk in (197, 577, 901):
    REACHABLE |= set(xtc(_Lk))
REACHABLE |= set(STC)

_NAME = re.compile(r"\b((?:attn|vit_attn|xattn|sattn)_\w*kernel|merge_parts_kernel)\b(<[^()]*>)?")


def attention_kernels(names):
    """Normalised attention kernel names ("attn_fwd_kernel<4,false>") among CUDA kernel names."""
    out = []
    for n in names:
        m = _NAME.search(n)
        if m:
            out.append(m.group(1) + re.sub(r"\s|\(int\)|\(bool\)", "", m.group(2) or ""))
    return out


def kernel_names(fn):
    """Names of the CUDA kernels fn() launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


# ------------------------------------------------------------------------------------------------ the case table
@dataclass
class Case:
    id: str
    kernels: tuple        # instantiations the forward + backward launch
    B: int
    H: int
    Lq: int
    Lk: int
    groups: tuple = None  # cross-attention: samples of each image (kv_offsets / kv_samples); None: self-attention
    tc: bool = True       # allow_tc
    table: bool = False   # relative-position table (ViT) together with the dense bias it gathers to
    bias: bool = False    # dense additive bias without a table
    kmask: bool = False
    drop: float = 0.0
    ds_dump: bool = False
    amp: float = 1.0      # std of q and k entries: the score std is amp^2 (scale 1/8, 64 dims)


R = lambda *g: tuple(g)
CASES = [
    # --- mma.sync, resident (allow_tc = 0, or shapes no tcgen05 kernel takes)
    Case("m_self197_bias_drop_ds", mma((4, 0), (4, 0), (4, 0)), 3, 2, 197, 197, tc=False, bias=True, drop=0.1, ds_dump=True),
    Case("m_text40_kmask_drop", mma((4, 0), (4, 0), (4, 0)), 5, 3, 40, 40, tc=False, kmask=True, drop=0.1),
    Case("m_self577_drop", mma((8, 0), (8, 0), (8, 0)), 1, 2, 577, 577, tc=False, drop=0.1),
    Case("m_vqa12x577_kmask_drop", mma((4, 0), (4, 0), (8, 0)), 6, 2, 12, 577, groups=R(2, 0, 3, 1), kmask=True, drop=0.1),
    Case("m_cross40x197_no_tc", mma((4, 0), (4, 0), (4, 0)), 9, 2, 40, 197, groups=R(7, 2), tc=False),
    # --- mma.sync, streaming
    Case("s_self901_bias_drop_ds", mma((8, 1), (8, 1), (8, 1)), 1, 2, 901, 901, bias=True, drop=0.1, ds_dump=True),
    Case("s_vqa12x901_kmask_drop", mma((4, 1), (4, 1), (8, 0)), 4, 3, 12, 901, groups=R(2, 0, 2), kmask=True, drop=0.1),
    Case("s_q901xk40", mma((8, 0), (8, 0), (4, 1)), 3, 2, 901, 40, groups=R(2, 1), drop=0.1),
    # --- tcgen05 ViT self-attention: every window with and without the table; B*H below / equal to / above 148 SMs
    Case("v4_table_ds", vit(4, True), 3, 2, 17, 17, table=True, ds_dump=True),
    Case("v4", vit(4, False), 2, 3, 17, 17),
    Case("v7_table_ds", vit(7, True), 3, 2, 50, 50, table=True, ds_dump=True),
    Case("v7", vit(7, False), 2, 2, 50, 50),
    Case("v12_table_ds", vit(12, True), 2, 3, 145, 145, table=True, ds_dump=True),
    Case("v12", vit(12, False), 3, 2, 145, 145),
    Case("v14_table_ds_148", vit(14, True), 37, 4, 197, 197, table=True, ds_dump=True),
    Case("v14_156", vit(14, False), 13, 12, 197, 197),
    Case("v14_table_amp8", vit(14, True), 2, 3, 197, 197, table=True, amp=2.83),
    Case("v24_table_ds", vit(24, True), 2, 2, 577, 577, table=True, ds_dump=True),
    Case("v24", vit(24, False), 1, 3, 577, 577),
    Case("v30_table_ds", vit(30, True), 1, 2, 901, 901, table=True, ds_dump=True),
    Case("v30", vit(30, False), 2, 1, 901, 901),
    # --- tcgen05 cross-attention, 40 text queries: groups of 1, GMAX = 6, more than 6 (chunked) and no sample at all
    Case("x197_groups_drop", xtc(197), 18, 4, 40, 197, groups=R(1, 6, 9, 0, 2), drop=0.1),
    Case("x197_148_items", xtc(197), 37, 4, 40, 197, groups=(1,) * 37),
    Case("x197_156_items_amp8", xtc(197), 26, 12, 40, 197, groups=(2, 1, 3) * 4 + (2,), amp=2.83),
    Case("x577_drop", xtc(577), 10, 2, 40, 577, groups=R(3, 0, 7), drop=0.1),
    Case("x901_drop", xtc(901), 5, 2, 40, 901, groups=R(1, 4, 0), drop=0.1),
    # --- tcgen05 text self-attention, three samples per tile: B not a multiple of 3; tiles below / equal to / above 148
    Case("t40_kmask_drop", STC, 5, 4, 40, 40, kmask=True, drop=0.1),
    Case("t40_148_tiles_kmask", STC, 111, 4, 40, 40, kmask=True),
    Case("t40_408_tiles_amp8", STC, 100, 12, 40, 40, amp=2.83, drop=0.1),
]
CASE_IDS = [c.id for c in CASES]
SEEN = {}


def _cross_index(groups, g):
    """kv_index for images with the given sample counts, samples in a shuffled order; kv_offsets / kv_samples (its CSR)."""
    kv_index = torch.cat([torch.full((n,), r, dtype=torch.int32) for r, n in enumerate(groups)])
    kv_index = kv_index[torch.randperm(len(kv_index), generator=g)]
    order = torch.argsort(kv_index.long(), stable=True).to(torch.int32)
    offs = torch.zeros(len(groups) + 1, dtype=torch.int32)
    offs[1:] = torch.cumsum(torch.tensor(groups), 0).to(torch.int32)
    return kv_index, offs, order


def make_inputs(c, seed):
    """Operands of a case (bf16 on the GPU) and the canary buffers of its outputs."""
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g)
    B, H, Lq, Lk = c.B, c.H, c.Lq, c.Lk
    D = H * 64
    t = dict()
    if c.groups is None:
        Bkv = B
        x = rnd(B * Lq, 3 * D)
        x[:, :2 * D] *= c.amp
        t["qkv"] = x.bfloat16().cuda()
        t["q"], t["k"], t["v"] = t["qkv"][:, :D], t["qkv"][:, D:2 * D], t["qkv"][:, 2 * D:]
        t["kv_index"] = None
    else:
        Bkv = len(c.groups)
        assert sum(c.groups) == B
        kv_index, offs, order = _cross_index(c.groups, g)
        t["kv_index"], t["kv_offsets"], t["kv_samples"] = kv_index.cuda(), offs.cuda(), order.cuda()
        t["q"] = (rnd(B * Lq, D) * c.amp).bfloat16().cuda()
        kv = rnd(Bkv * Lk, 2 * D)
        kv[:, :D] *= c.amp
        t["kv"] = kv.bfloat16().cuda()
        t["k"], t["v"] = t["kv"][:, :D], t["kv"][:, D:]
    t["Bkv"] = Bkv
    t["dout"] = rnd(B * Lq, D).bfloat16().cuda()
    t["bias_ld"] = _r8(Lk)
    if c.table:
        from xfm_b200.encoders import closed_form_rel_index
        W = math.isqrt(Lk - 1)
        table = rnd((2 * W - 1) ** 2 + 3, H)
        t["table"] = table.cuda()
        t["dense"] = table[closed_form_rel_index(W).view(-1)].view(Lq, Lk, H).permute(2, 0, 1).contiguous().cuda()
    elif c.bias:
        t["dense"] = rnd(H, Lq, Lk).cuda()
    if "dense" in t:
        t["bias"] = torch.zeros(H, Lq, t["bias_ld"], device="cuda")
        t["bias"][..., :Lk] = t["dense"]
    if c.kmask:
        t["kmask"] = torch.where(torch.rand(B, Lk, generator=g) < 0.2, -10000.0, 0.0).cuda()
    # outputs inside canaries: out with a row stride wider than its columns, lse / delta / ds as whole tensors, dq / dk / dv
    # as the column slices of one dqkv (self-attention) or dq + dkv (cross-attention) buffer
    t["out"] = Buf(B * Lq, D, D + 8, BF16)
    t["lse"] = Buf(1, B * H * Lq, B * H * Lq, F32)
    t["delta"] = Buf(1, B * H * Lq, B * H * Lq, F32)
    if c.groups is None:
        t["dqkv"] = Buf(B * Lq, 3 * D, 3 * D + 8, BF16)
        v = t["dqkv"].view
        t["dq"], t["dk"], t["dv"] = v[:, :D], v[:, D:2 * D], v[:, 2 * D:]
        t["grad_bufs"] = [(t["dqkv"], [t["dq"], t["dk"], t["dv"]])]
    else:
        t["dqb"] = Buf(B * Lq, D, D + 8, BF16)
        t["dkv"] = Buf(Bkv * Lk, 2 * D, 2 * D + 8, BF16)
        t["dq"], t["dk"], t["dv"] = t["dqb"].view, t["dkv"].view[:, :D], t["dkv"].view[:, D:]
        t["grad_bufs"] = [(t["dqb"], [t["dq"]]), (t["dkv"], [t["dk"], t["dv"]])]
    if c.ds_dump:
        t["ds_ld"] = _r8(Lk)
        t["ds"] = Buf(1, B * H * Lq * t["ds_ld"], B * H * Lq * t["ds_ld"], BF16)
        if not c.tc or "vit" not in c.kernels[0]:   # the mma.sync kernels leave the padding columns to the caller
            t["ds"].view.view(B, H, Lq, t["ds_ld"])[..., Lk:] = 0
    return t


def _params(L, c, t, seed):
    p = L.AttnParams()
    p.q, p.k, p.v = t["q"].data_ptr(), t["k"].data_ptr(), t["v"].data_ptr()
    p.q_stride, p.k_stride, p.v_stride = t["q"].stride(0), t["k"].stride(0), t["v"].stride(0)
    p.B, p.H, p.Lq, p.Lk, p.head_dim, p.Bkv = c.B, c.H, c.Lq, c.Lk, 64, t["Bkv"]
    p.scale, p.dropout_p, p.dropout_seed = SCALE, c.drop, seed
    if "bias" in t:
        p.bias, p.bias_ld = t["bias"].data_ptr(), t["bias_ld"]
    if "table" in t:
        p.rel_table, p.rel_window = t["table"].data_ptr(), math.isqrt(c.Lk - 1)
    if "kmask" in t:
        p.kmask = t["kmask"].data_ptr()
    if t["kv_index"] is not None:
        p.kv_index, p.kv_offsets, p.kv_samples = (t[k].data_ptr() for k in ("kv_index", "kv_offsets", "kv_samples"))
    p.allow_tc = int(c.tc)
    return p


def run(L, c, t, seed):
    """Forward then backward of the case with every output inside its canary buffer."""
    for k in ("out", "lse", "delta", "ds", "dqb", "dkv", "dqkv"):
        if k in t:
            t[k].snapshot()
    p = _params(L, c, t, seed)
    p.out, p.o_stride, p.lse = t["out"].view.data_ptr(), t["out"].view.stride(0), t["lse"].view.data_ptr()
    nb = L.load().xfm_attention_fwd_parts(C.byref(p))
    if nb:
        parts = (torch.empty((nb, c.B * c.Lq, c.H * 64), dtype=BF16, device="cuda"),
                 torch.empty((nb, c.B, c.H, c.Lq), dtype=F32, device="cuda"))
        p.part_out, p.part_lse = parts[0].data_ptr(), parts[1].data_ptr()
    L.check(L.lib().xfm_attention_fwd(C.byref(p), L.stream_ptr()), "xfm_attention_fwd")
    p.dout, p.do_stride, p.delta = t["dout"].data_ptr(), t["dout"].stride(0), t["delta"].view.data_ptr()
    p.dq, p.dk, p.dv = t["dq"].data_ptr(), t["dk"].data_ptr(), t["dv"].data_ptr()
    p.dq_stride, p.dk_stride, p.dv_stride = t["dq"].stride(0), t["dk"].stride(0), t["dv"].stride(0)
    if "ds" in t:
        p.ds_dump, p.ds_ld = t["ds"].view.data_ptr(), t["ds_ld"]
    L.check(L.lib().xfm_attention_bwd(C.byref(p), L.stream_ptr()), "xfm_attention_bwd")


def keep_mask(c, seed):
    """[B, H, Lq, Lk] kept set of the case's dropout (None without dropout)."""
    if not c.drop:
        return None
    return torch.from_numpy(DM.keep(seed, DM.attention_index(c.B, c.H, c.Lq, c.Lk), c.drop)).cuda()


def _heads(x, n, L, H):
    return x.double().reshape(n, L, H, 64).permute(0, 2, 1, 3)


def reference(c, t, keep):
    """fp64 forward and backward with their magnitude tensors.  The backward reference takes delta from the bf16 `out` the
    backward is given, as the kernels do."""
    B, H, Lq, Lk, Bkv = c.B, c.H, c.Lq, c.Lk, t["Bkv"]
    q = _heads(t["q"], B, Lq, H)
    kr, vr = _heads(t["k"], Bkv, Lk, H), _heads(t["v"], Bkv, Lk, H)
    idx = t["kv_index"].long() if t["kv_index"] is not None else torch.arange(B, device=q.device)
    k, v = kr[idx], vr[idx]
    add = torch.zeros(1, 1, 1, 1, dtype=torch.float64, device=q.device)
    if "dense" in t:
        add = add + t["dense"].double()[None]
    if "kmask" in t:
        add = add + t["kmask"].double()[:, None, None, :]
    raw = SCALE * (q @ k.transpose(-1, -2))
    s = raw + add
    P = torch.softmax(s, -1)
    pf = float(np.float32(c.drop))
    kf = keep.double() / (1.0 - pf) if keep is not None else 1.0
    Pt = P * kf
    r = dict(out=Pt @ v, lse=torch.logsumexp(s, -1))
    m = dict(out=Pt.abs() @ v.abs(), lse=(P * (SCALE * (q.abs() @ k.abs().transpose(-1, -2)) + add.abs())).sum(-1) + 1.0)
    do = _heads(t["dout"], B, Lq, H)
    o_given = _heads(t["out"].view, B, Lq, H)
    delta = (do * o_given).sum(-1, keepdim=True)
    dP = do @ v.transpose(-1, -2)
    dS = P * (dP * kf - delta)
    G = P * ((do.abs() @ v.abs().transpose(-1, -2)) / (1.0 - pf) + delta.abs())
    r["delta"], m["delta"] = delta[..., 0], (do.abs() * o_given.abs()).sum(-1)
    r["ds"], m["ds"] = dS, G
    r["dq"], m["dq"] = SCALE * dS @ k, SCALE * G @ k.abs()
    zk = torch.zeros_like(kr)
    r["dk"] = zk.index_add(0, idx, SCALE * dS.transpose(-1, -2) @ q)
    m["dk"] = zk.index_add(0, idx, SCALE * G.transpose(-1, -2) @ q.abs())
    r["dv"] = zk.index_add(0, idx, Pt.transpose(-1, -2) @ do)
    m["dv"] = zk.index_add(0, idx, Pt.abs().transpose(-1, -2) @ do.abs())
    return r, m


def got(c, t):
    B, H, Lq, Lk, Bkv = c.B, c.H, c.Lq, c.Lk, t["Bkv"]
    g = dict(out=_heads(t["out"].view, B, Lq, H), lse=t["lse"].view.double().view(B, H, Lq),
             delta=t["delta"].view.double().view(B, H, Lq), dq=_heads(t["dq"], B, Lq, H),
             dk=_heads(t["dk"], Bkv, Lk, H), dv=_heads(t["dv"], Bkv, Lk, H))
    if "ds" in t:
        ds = t["ds"].view.double().view(B, H, Lq, t["ds_ld"])
        g["ds"], g["ds_pad"] = ds[..., :Lk], ds[..., Lk:]
    return g


def n_round(c, name):
    """bf16 roundings of partial sums: dQ of a key-block tcgen05 backward is reduce-added once per key block; dK / dV of
    an image whose samples the tcgen05 cross-attention backward takes in chunks of 3, once per chunk."""
    tc_bwd = any("tc_kernel" in k for k in c.kernels)
    if name == "dq" and tc_bwd:
        return _nb(c.Lk)
    if name in ("dk", "dv") and tc_bwd and c.groups is not None:
        return max((n + 2) // 3 for n in c.groups)
    return 0


CONST = dict(out=C_OUT, lse=C_LSE, dq=C_GRAD, dk=C_GRAD, dv=C_GRAD, ds=C_DS)


def _ratio(err, bnd):
    """err / bound per element; 0 where both are 0 (dK / dV of an image without samples are exactly 0)."""
    return torch.where(bnd > 0, err / bnd.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))


@pytest.mark.parametrize("c", CASES, ids=CASE_IDS)
def test_attention_case(lib, record, c):
    """One row of CASES: the kernels it names run, every output is within its per-element bound of the fp64 reference,
    and no byte outside the outputs' views changes."""
    seed = 101 + CASE_IDS.index(c.id)
    t = make_inputs(c, seed)
    names = attention_kernels(kernel_names(lambda: run(lib, c, t, seed)))
    SEEN[c.id] = set(names)
    print(c.id, sorted(set(names)))
    assert set(names) == set(c.kernels), (sorted(set(names)), sorted(c.kernels))
    for k in ("out", "lse", "delta", "ds"):
        if k in t:
            assert t[k].outside_unchanged(), k + " written outside its view"
    for b, views in t["grad_bufs"]:
        assert b.outside_unchanged(views), "dq / dk / dv written outside their column slices"
    r, m = reference(c, t, keep_mask(c, seed))
    g = got(c, t)
    report, worst = {}, {}
    for name in ("out", "lse", "dq", "dk", "dv", "ds"):
        if name not in g:
            continue
        assert torch.isfinite(g[name]).all(), name + " has non-finite elements"
        err = (g[name] - r[name]).abs()
        rest = U_BF16 * (r[name].abs() + n_round(c, name) * m[name]) if name != "lse" else 0.0
        bnd = CONST[name] * m[name] + rest
        worst[name] = float(_ratio(err, bnd).max())
        report[name] = float(((err - rest) / m[name].clamp_min(1e-300)).max())   # the smallest C this row would pass
    # delta: a 64-term fp32 dot product of the given bf16 out and dO
    err = (g["delta"] - r["delta"]).abs()
    worst["delta"] = float(_ratio(err, 2.0 ** -17 * m["delta"]).max())
    if "ds_pad" in g:
        assert float(g["ds_pad"].abs().max()) == 0.0, "dS padding columns are not zero"
    record("attention_case", case=c.id, worst_ratio=worst, c_needed=report)
    print(c.id, "c_needed", {k: "2^%.1f" % math.log2(v) if v > 0 else 0 for k, v in report.items()})
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, (bad, report)


def test_every_instantiation_is_reached():
    """The rows of CASES name every attention instantiation the dispatch can launch, and (when they all ran) ran them."""
    declared = set().union(*(set(c.kernels) for c in CASES))
    assert declared == REACHABLE, (sorted(REACHABLE - declared), sorted(declared - REACHABLE))
    if len(SEEN) == len(CASES):
        missed = REACHABLE - set().union(*SEEN.values())
        print("attention instantiations reached:", len(REACHABLE) - len(missed), "of", len(REACHABLE), "missed:", sorted(missed))
        assert not missed, sorted(missed)


# ------------------------------------------------------------------------------------------------ exact dropout masks
def test_dropout_apply_is_the_oracle(lib):
    """The oracle's hash is the device's: dropout_apply on ones keeps exactly the oracle's element set."""
    n, p, seed = 1 << 20, 0.1, (7 << 32) + 12345
    y = lib.dropout_apply(torch.ones(n, dtype=torch.float32, device="cuda"), p, seed)
    kept = (y != 0).cpu().numpy()
    assert np.array_equal(kept, DM.keep(seed, np.arange(n), p))
    assert float(y[y != 0].float().min()) == float(torch.tensor(1.0 / (1.0 - np.float32(p))).bfloat16())


@dataclass
class Probe:
    id: str
    B: int
    H: int
    Lq: int
    Lk: int
    groups: tuple = None
    tc: bool = True


PROBES = [
    Probe("mma_resident_197", 2, 2, 197, 197, tc=False),            # <4, false> x 3
    Probe("mma_resident_577", 1, 2, 577, 577, tc=False),            # <8, false> x 3
    Probe("mma_text40", 4, 2, 40, 40, tc=False),                     # <4, false> x 3
    Probe("mma_stream_901", 1, 2, 901, 901),                        # <8, true> x 3
    Probe("mma_stream_12x901", 3, 2, 12, 901, groups=(2, 1)),       # fwd / dq <4, true>, dkv <8, false>
    Probe("mma_stream_dkv_901x40", 2, 2, 901, 40, groups=(2,)),     # dkv <4, true>
    Probe("xtc_197", 12, 2, 40, 197, groups=(1, 9, 0, 2)),
    Probe("xtc_577", 8, 2, 40, 577, groups=(7, 1)),
    Probe("xtc_901", 4, 2, 40, 901, groups=(3, 0, 1)),
    Probe("stc_40", 5, 3, 40, 40),
]


def _probe_run(L, pr, q, k, v, dout, out_given, p, seed, ix, bwd):
    """Forward (and backward) of a probe; returns out, or (dq, dk, dv) of the backward."""
    kw = dict(Bkv=ix[3], allow_tc=pr.tc, dropout_p=p, dropout_seed=seed)
    if ix[0] is not None:
        kw.update(kv_index=ix[0], kv_offsets=ix[1], kv_samples=ix[2])
    out, lse = L.attention_fwd(q, k, v, pr.B, pr.H, pr.Lq, pr.Lk, SCALE, **kw)
    if not bwd:
        return out
    dq = torch.empty_like(q)
    dk, dv = torch.empty_like(k), torch.empty_like(v)
    L.attention_bwd(dout, q, k, v, out if out_given is None else out_given, lse, pr.B, pr.H, pr.Lq, pr.Lk, SCALE, dq, dk, dv,
                    **kw)
    return dq, dk, dv


@pytest.mark.parametrize("pr", PROBES, ids=[x.id for x in PROBES])
def test_dropout_mask_is_the_hash(lib, pr):
    """Each kernel's kept set, recovered bit for bit, is the hash of element ((b H + h) Lq + q) LKE + key.  q = 0 makes
    P = 1/Lk.  Forward: V_j = e_(j - 64w) on the key window w, zero elsewhere, so out[i, d] != 0 iff key 64w + d is kept.
    dV: dO_i = e_(i - 64w) on a query window, for one sample of each image at a time.  dQ: V_j = dO_i = e_0 and out = 0
    (delta = 0), K_j one-hot on a key window: dQ[i, d] = scale P / (1 - p) when key 64w + d is kept, else 0.  Head h takes
    window (h + call) mod n, so the calls together cover every key of every head."""
    B, H, Lq, Lk, p, seed = pr.B, pr.H, pr.Lq, pr.Lk, 0.25, 4242 + PROBES.index(pr)
    D = H * 64
    dev = "cuda"
    if pr.groups is None:
        Bkv, ix, samples = B, (None, None, None, B), [[b] for b in range(B)]
    else:
        Bkv = len(pr.groups)
        kv_index, offs, order = _cross_index(pr.groups, torch.Generator().manual_seed(seed))
        ix = (kv_index.to(dev), offs.to(dev), order.to(dev), Bkv)
        samples = [order[offs[r]:offs[r + 1]].tolist() for r in range(Bkv)]
    want = DM.keep(seed, DM.attention_index(B, H, Lq, Lk), p)
    q = torch.zeros(B * Lq, D, dtype=BF16, device=dev)
    eye = torch.eye(64, dtype=BF16, device=dev)

    def one_hot_rows(n_rows, L, win_of_head, sel=None):
        """[n_rows * L, D]: row j of head h is e_(j - 64 w) inside window w = win_of_head[h], zero elsewhere."""
        x = torch.zeros(n_rows, L, H, 64, dtype=BF16, device=dev)
        for h, w in enumerate(win_of_head):
            n = min(64, L - 64 * w)
            rows = x[:, 64 * w:64 * w + n, h]
            rows.copy_(eye[:n].expand(rows.shape))
        if sel is not None:
            off = torch.ones(n_rows, dtype=torch.bool, device=dev)
            off[sel] = False
            x[off] = 0
        return x.view(n_rows * L, D)

    def e0(n):
        x = torch.zeros(n, D, dtype=BF16, device=dev)
        x.view(n, H, 64)[:, :, 0] = 1
        return x

    got = {k: np.zeros((B, H, Lq, Lk), dtype=np.int8) - 1 for k in ("fwd", "dv", "dq")}
    nk, nq = (Lk + 63) // 64, (Lq + 63) // 64
    for call in range(nk):   # forward and dQ: key windows
        wins = [(h + call) % nk for h in range(H)]
        onehot = one_hot_rows(Bkv, Lk, wins)
        zero_kv = torch.zeros_like(onehot)
        out = _probe_run(lib, pr, q, zero_kv, onehot, None, None, p, seed, ix, False)
        dq, _, _ = _probe_run(lib, pr, q, onehot, e0(Bkv * Lk), e0(B * Lq), torch.zeros(B * Lq, D, dtype=BF16, device=dev), p,
                              seed, ix, True)
        o4 = (out.view(B, Lq, H, 64) != 0).cpu().numpy()
        g4 = (dq.view(B, Lq, H, 64) != 0).cpu().numpy()
        for h, w in enumerate(wins):
            n = min(64, Lk - 64 * w)
            got["fwd"][:, h, :, 64 * w:64 * w + n] = o4[:, :, h, :n]
            got["dq"][:, h, :, 64 * w:64 * w + n] = g4[:, :, h, :n]
    for call in range(nq):   # dV: query windows, one sample of each image per call
        wins = [(h + call) % nq for h in range(H)]
        for rank in range(max(len(s) for s in samples)):
            sel = [s[rank] for s in samples if rank < len(s)]
            do = one_hot_rows(B, Lq, wins, torch.tensor(sel, device=dev))
            kv0 = torch.zeros(Bkv * Lk, D, dtype=BF16, device=dev)
            _, _, dv = _probe_run(lib, pr, q, kv0, kv0, do, None, p, seed, ix, True)
            d4 = (dv.view(Bkv, Lk, H, 64) != 0).cpu().numpy()
            for r, s in enumerate(samples):
                if rank >= len(s):
                    continue
                for h, w in enumerate(wins):
                    n = min(64, Lq - 64 * w)
                    got["dv"][s[rank], h, 64 * w:64 * w + n, :] = d4[r, :, h, :n].T
    for k, g in got.items():
        assert (g >= 0).all(), k + ": probe left elements unrecovered"
        diff = int((g.astype(bool) != want).sum())
        assert diff == 0, "%s: %d of %d mask bits differ from the hash" % (k, diff, want.size)


# ------------------------------------------------------------------------------------------------ argument checks
def test_bwd_rejects_kv_index_without_csr(lib):
    """kv_index without kv_offsets / kv_samples: dK / dV would be identity-mapped; the backward refuses before any launch."""
    B, Bkv, H, Lq, Lk = 4, 2, 2, 40, 197
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(3)
    q = torch.randn(B * Lq, D, device="cuda", generator=g).bfloat16()
    kv = torch.randn(Bkv * Lk, 2 * D, device="cuda", generator=g).bfloat16()
    do = torch.randn(B * Lq, D, device="cuda", generator=g).bfloat16()
    kv_index = torch.tensor([0, 1, 0, 1], dtype=torch.int32, device="cuda")
    out, lse = lib.attention_fwd(q, kv[:, :D], kv[:, D:], B, H, Lq, Lk, SCALE, Bkv=Bkv, kv_index=kv_index)
    dq, dkv = Buf(B * Lq, D, D, BF16), Buf(Bkv * Lk, 2 * D, 2 * D, BF16)
    torch.cuda.synchronize()
    dq.snapshot()
    dkv.snapshot()
    for tc in (True, False):
        with pytest.raises(RuntimeError, match="kv_offsets"):
            lib.attention_bwd(do, q, kv[:, :D], kv[:, D:], out, lse, B, H, Lq, Lk, SCALE, dq.view, dkv.view[:, :D],
                              dkv.view[:, D:], Bkv=Bkv, kv_index=kv_index, allow_tc=tc)
    torch.cuda.synchronize()
    assert dq.unchanged() and dkv.unchanged()
