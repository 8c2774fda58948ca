"""xfm_gemm_bf16 and xfm_sgemm_f32 against an fp64 reference of the same operation, path by path.

Every case of CASES is chosen to reach one kernel instantiation and epilogue path of gemm.cu (the `kernel` and `path`
columns, worked out from gemm_bf16 / launch_gemm_pair); test_every_instantiation_is_reached checks the instantiation of
each row with the profiler.  The reference is the fp64 product of the same bf16 operands followed by the epilogue in the
order of include/xfm_b200.h.  Errors are bounded per element (bound() below), never relative to the largest value of the
matrix, so a wrong column with a small LayerScale gamma, a wrong row group with a small DropPath scale or a wrong ragged
tile cannot hide behind large values elsewhere.  Outputs live inside larger canary-filled buffers and every byte outside
[M, N] must survive the call.
"""
import itertools
import math
from dataclasses import dataclass

import numpy as np
import pytest
import torch
from canary import Buf

from oracle.dropout_mask import keep

pytestmark = pytest.mark.gpu

# Accumulation error of the tcgen05 GEMM, per element: |acc - exact| <= C_ACC * (|A|.|B|)_ij (the other terms: bound()).
# The smallest power of two that every case below passes on a B200 (NVIDIA B200, 1000 W power limit): the largest C_ACC a
# case needed was 6.5e-7 = 2^-20.5 (p_tt_wgrad_fc1, K = 18912 split in two), every case with K <= 1152 needed < 2^-22.
C_ACC = 2.0 ** -20
GELU_SLOPE = 1.13   # max |gelu'(x)| = gelu'(sqrt 2) = 1.1290
U32 = 2.0 ** -24    # fp32 unit roundoff
E_ERF = 2.0 ** -21  # |gelu_fast - gelu| <= E_ERF |x| and |gelu_grad_fast - gelu'| <= E_ERF (common.cuh erf_core: A&S 7.1.26)


@pytest.fixture(scope="module")
def lib():
    from xfm_b200 import lib as L

    L.lib()
    L.seed_salt_set(0)   # dropout masks below depend on dropout_seed only
    return L


def _r8(x):
    return (x + 7) // 8 * 8


def keep_mask(M, N, seed, p):
    """The dropout mask of an [M, N] epilogue: element row * N + col of common.cuh's hash."""
    return torch.from_numpy(keep(seed, np.arange(M * N), p).reshape(M, N))


# ------------------------------------------------------------------------------------------------ the case matrix
@dataclass
class Case:
    id: str
    family: str       # single | pair | epilogue
    kernel: str       # instantiation the dispatch must pick: single<BLOCK_N,A_MN,B_MN> or pair<A_MN,B_MN,EPI>
    path: str         # what else of the dispatch the case targets
    M: int
    N: int
    K: int
    bn: int = 512     # block_n: 512 forces the CTA-pair kernel
    a_t: bool = False
    b_t: bool = False
    out: torch.dtype = torch.bfloat16
    bias: bool = False
    aux_out: bool = False
    act: int = 0
    col_scale: bool = False
    rpg: int = 0      # rows_per_group of row_group_scale (0: none)
    drop: float = 0.0
    res: torch.dtype = None
    acc: bool = False
    split: int = 1
    ldc: int = 0      # 0: round8(N) + 8
    c_off: int = 0    # C's element offset inside its buffer (1 f32 / 2 bf16 = 4 bytes: not 8 / 16-byte aligned)
    aux_ld: int = 0   # 0: round8(N) + 16
    lda: int = 0      # 0: round8 of the stored row length


F32, BF16 = torch.float32, torch.bfloat16
# Single-CTA kernel: block_n 64 / 128 / 256 (gemm_bf16 switch).  epi_mode (gemm.cu gemm_bf16): 0 = bf16 out, act <= 1, no
# scales / dropout / residual; 1 = the same with act 2 and no aux_out; 2 = everything else.  vec_ok = 0 (scalar epilogue)
# when C is not 4-byte (bf16) / 8-byte (f32) aligned or ldc is odd.
# CTA-pair kernel (launch_gemm_pair): EPI 1 = mode 2, f32 out, no accumulate, no split, act 0, N % 32 == 0, 16-byte aligned
# C / residual (f32) / aux_out; EPI 2 = mode 1, split 1, N % 32 == 0, aligned C / aux_in, ldc % 8 == 0; EPI 0 otherwise, with
# the bf16 TMA store (tma_epi = 1) for modes 0 / 1 at split 1 with 16-byte aligned C / aux pointers and ldc % 8 == 0.
# N-fastest tile order: split 1, more than one N tile, A > 40 MB and B <= 16 MB (always for EPI 1).
CASES = [
    # --- single-CTA, every BLOCK_N x layout; ragged M (1, 127, 129), N (8, 40, 1000), K (8, 40, 72, 200)
    Case("s64_kk_bias_ragged", "single", "single<64,0,0>", "mode 0 with a bias, ragged M/N/K", 127, 40, 72, bn=64, bias=True),
    Case("s64_tt_f32", "single", "single<64,1,1>", "mode 2 plain f32, BLOCK_N 64 with MN-major operands",
         129, 1000, 200, bn=64, a_t=True, b_t=True, out=F32),
    Case("s64_kt_dgelu_tiny", "single", "single<64,0,1>", "mode 1, M = 1, N = 8, K shorter than one k-block",
         1, 8, 8, bn=64, b_t=True, act=2),
    Case("s64_tk_gelu_aux", "single", "single<64,1,0>", "mode 0, GELU + saved pre-activation, K = 40",
         200, 100, 40, bn=64, a_t=True, bias=True, act=1, aux_out=True),
    Case("s128_kk_tanh", "single", "single<128,0,0>", "mode 2, tanh + aux_out + col_scale, f32 out",
         129, 1000, 200, bn=128, out=F32, bias=True, aux_out=True, act=3, col_scale=True),
    Case("s128_kt_dgelu_bias", "single", "single<128,0,1>", "mode 1, dGELU with a bias", 127, 40, 72, bn=128, b_t=True,
         bias=True, act=2),
    Case("s128_tk_res_bf16", "single", "single<128,1,0>", "mode 2, bf16 residual, bf16 out", 256, 384, 256, bn=128,
         a_t=True, bias=True, res=BF16),
    Case("s128_tt_splitk_scales", "single", "single<128,1,1>", "mode 2, split-K 3 accumulate, col_scale, rows_per_group 17, "
         "dropout", 300, 264, 520, bn=128, a_t=True, b_t=True, out=F32, acc=True, split=3, col_scale=True, rpg=17, drop=0.1),
    Case("s256_kk_odd_ldc", "single", "single<256,0,0>", "mode 0, scalar epilogue: odd ldc and odd aux_out ld",
         300, 1000, 200, bn=256, bias=True, act=1, aux_out=True, ldc=1011, aux_ld=1003),
    Case("s256_kt_offset_c", "single", "single<256,0,1>", "mode 2, scalar epilogue: C at a 4-byte offset, rows_per_group 1",
         129, 520, 8, bn=256, b_t=True, out=F32, col_scale=True, rpg=1, c_off=1),
    Case("s256_tk_drop_res", "single", "single<256,1,0>", "mode 2, dropout + f32 residual, rows_per_group 577",
         1200, 264, 128, bn=256, a_t=True, out=F32, bias=True, rpg=577, drop=0.1, res=F32),
    Case("s256_tt_acc", "single", "single<256,1,1>", "mode 2, accumulate (split 1) onto random C, rows_per_group 197",
         600, 512, 256, bn=256, a_t=True, b_t=True, out=F32, acc=True, rpg=197),
    # --- CTA pair, every layout x EPI 0 / 1 / 2
    Case("p_kk_tma_store", "pair", "pair<0,0,0>", "bf16 TMA store, 5 M tiles (odd), N % 32 != 0 and N % 256 != 0",
         640, 520, 192, bias=True, act=1, aux_out=True),
    Case("p_kk_no_tma_store", "pair", "pair<0,0,0>", "mode 0 generic epilogue: C at a 4-byte offset rules out the TMA store",
         384, 264, 128, bias=True, act=1, c_off=2),
    Case("p_kt_generic", "pair", "pair<0,1,0>", "mode 2 generic epilogue: C at a 4-byte offset (no TMA store), tanh, "
         "bf16 residual", 384, 300, 128, b_t=True, bias=True, act=3, res=BF16, c_off=2),
    Case("p_tk_empty_slice", "pair", "pair<1,0,0>", "split-K 3 over 4 k-blocks: the third slice is empty",
         640, 264, 256, a_t=True, out=F32, acc=True, split=3),
    Case("p_kk_f32", "pair", "pair<0,0,1>", "f32 TMA epilogue, bias only, 9 M tiles", 1152, 768, 64, out=F32, bias=True),
    Case("p_kt_f32_res", "pair", "pair<0,1,1>", "f32 TMA epilogue, col_scale + f32 residual", 384, 256, 256, b_t=True,
         out=F32, col_scale=True, res=F32),
    Case("p_tk_f32_all", "pair", "pair<1,0,1>", "f32 TMA epilogue, bias + aux_out + col_scale + rows_per_group 197 + "
         "f32 residual", 640, 512, 192, a_t=True, out=F32, bias=True, aux_out=True, col_scale=True, rpg=197, res=F32),
    Case("p_tt_f32_drop", "pair", "pair<1,1,1>", "f32 TMA epilogue, dropout + rows_per_group 17", 640, 288, 128, a_t=True,
         b_t=True, out=F32, rpg=17, drop=0.1),
    Case("p_kk_dgelu", "pair", "pair<0,0,2>", "dGELU TMA epilogue, ragged K", 640, 544, 72, act=2),
    Case("p_kt_dgelu_bias", "pair", "pair<0,1,2>", "dGELU TMA epilogue with a bias", 640, 800, 136, b_t=True, bias=True,
         act=2),
    Case("p_tk_dgelu", "pair", "pair<1,0,2>", "dGELU TMA epilogue with a bias, 3 M tiles", 384, 256, 128, a_t=True,
         bias=True, act=2),
    Case("p_tt_dgelu", "pair", "pair<1,1,2>", "dGELU TMA epilogue, 7 M tiles", 896, 320, 200, a_t=True, b_t=True, bias=True,
         act=2),
    # weight gradients (blocks.wgrad): fc1 3072 x 768 and qkv 2304 x 768 over T = 18912 tokens; the tied word-embedding
    # gradient scaled down (M = 4099 rows, MN-major A with the padded row stride of the logits)
    Case("p_tt_wgrad_fc1", "pair", "pair<1,1,0>", "split-K wgrad", 3072, 768, 18912, a_t=True, b_t=True, out=F32, acc=True,
         split=-1),
    Case("p_tt_wgrad_qkv", "pair", "pair<1,1,0>", "split-K wgrad", 2304, 768, 18912, a_t=True, b_t=True, out=F32, acc=True,
         split=-1),
    Case("p_tt_wgrad_word", "pair", "pair<1,1,0>", "wgrad, M % 8 != 0, lda 4104", 4099, 768, 1024, a_t=True, b_t=True,
         out=F32, acc=True, split=-1, lda=4104),
    # N-fastest tile order: A = 20480 x 1152 bf16 = 47 MB > 40 MB
    Case("p_kk_nfast_gelu", "pair", "pair<0,0,0>", "N-fastest, bf16 TMA store, GELU + aux_out", 20480, 768, 1152, bias=True,
         act=1, aux_out=True),
    Case("p_kt_nfast_dgelu", "pair", "pair<0,1,2>", "N-fastest, dGELU TMA epilogue", 20480, 768, 1152, b_t=True, bias=True,
         act=2),
    # --- epilogue features not covered above
    Case("e_gelu_no_bias_strided", "epilogue", "single<128,0,0>", "mode 0, GELU without bias, strided C", 257, 264, 128,
         bn=128, act=1, ldc=320),
    Case("e_tanh_bf16", "epilogue", "single<64,0,0>", "mode 2, tanh into bf16 output", 200, 96, 136, bn=64, bias=True, act=3),
    Case("e_dgelu_aux_out", "epilogue", "single<128,0,1>", "mode 2: dGELU together with aux_out, f32 out", 160, 200, 128,
         bn=128, b_t=True, out=F32, bias=True, act=2, aux_out=True),
    Case("e_rpg1_pair_generic", "epilogue", "pair<0,0,0>", "mode 2 bf16 out: rows_per_group 1 + col_scale + dropout",
         384, 264, 128, col_scale=True, rpg=1, drop=0.1),
    Case("e_rpg577_pair_f32", "epilogue", "pair<0,0,1>", "f32 TMA epilogue, rows_per_group 577 straddles 32-row blocks",
         1400, 256, 128, out=F32, rpg=577, col_scale=True, bias=True),
]
CASE_IDS = [c.id for c in CASES]


def _split_of(c):
    if c.split >= 0:
        return c.split
    from xfm_b200.blocks import _split_k   # the factor blocks.wgrad picks for this shape
    return _split_k(((c.M + 255) // 256) * ((c.N + 255) // 256), 74, (c.K + 63) // 64)


def launch(L, c, seed, split=None):
    """Build the case's operands inside canary buffers, run xfm_gemm_bf16 once and return what the reference needs."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g)
    M, N, K = c.M, c.N, c.K
    a = Buf(K, M, c.lda or _r8(M), BF16) if c.a_t else Buf(M, K, c.lda or _r8(K), BF16)
    a.view.copy_(rnd(*a.shape))
    b = Buf(K, N, _r8(N), BF16) if c.b_t else Buf(N, K, _r8(K), BF16)
    b.view.copy_(rnd(*b.shape) * K ** -0.5)
    t = dict(A=a.view.t() if c.a_t else a.view, B=b.view.t() if c.b_t else b.view)
    kw = {}
    if c.bias:
        t["bias"] = kw["bias"] = rnd(N) * 0.5
    if c.act:
        kw["act"] = c.act
    if c.act == 2:
        aux_in = Buf(M, N, _r8(N) + 8, BF16)
        aux_in.view.copy_(rnd(M, N))
        t["aux_in"] = kw["aux_in"] = aux_in.view
    if c.col_scale:   # LayerScale gamma: magnitudes 0.01 .. 2, both signs
        u = torch.rand(N, device="cuda", generator=g)
        t["col_scale"] = kw["col_scale"] = torch.where(rnd(N) < 0, -1.0, 1.0) * 10.0 ** (2.3 * u - 2.0)
    if c.rpg:         # per-sample scales 0.05 .. 1.5
        ng = (M + c.rpg - 1) // c.rpg
        t["rgs"] = kw["row_group_scale"] = 0.05 + 1.45 * torch.rand(ng, device="cuda", generator=g)
        kw["rows_per_group"] = c.rpg
    if c.drop:
        kw["dropout_p"], kw["dropout_seed"] = c.drop, seed
    if c.res is not None:
        res = Buf(M, N, _r8(N) + 8, c.res)
        res.view.copy_(rnd(M, N))
        t["res"] = kw["residual"] = res.view
    out = Buf(M, N, c.ldc or _r8(N) + 8, c.out, c.c_off)
    if c.acc:
        out.view.copy_(rnd(M, N))
        t["C0"] = out.view.double()
    if c.aux_out:
        t["aux_out"] = Buf(M, N, c.aux_ld or _r8(N) + 16, BF16)
        kw["aux_out"] = t["aux_out"].view
        t["aux_out"].snapshot()
    out.snapshot()
    t["out"] = out
    L.gemm(a.view, b.view, a_t=c.a_t, b_t=c.b_t, out=out.view, accumulate=c.acc,
           split_k=_split_of(c) if split is None else split, block_n=c.bn, **kw)
    return t


def _gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _dgelu(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def epilogue64(acc, t, c, keep):
    """The header's epilogue in fp64: returns (R, z, gain, act_err): z = acc + bias, gain bounds |dR / d acc| per element,
    act_err bounds the kernel's approximation of the activation (already scaled like R)."""
    z = acc + t["bias"].double() if "bias" in t else acc
    if c.act == 1:
        y, gain, act_err = _gelu(z), GELU_SLOPE, E_ERF * z.abs()
    elif c.act == 2:
        d = _dgelu(t["aux_in"].double())
        y, gain, act_err = z * d, d.abs(), E_ERF * z.abs()
    elif c.act == 3:
        y, gain, act_err = torch.tanh(z), 1.0, 4 * U32 * torch.tanh(z).abs()
    else:
        y, gain, act_err = z, 1.0, 0.0
    post = torch.ones_like(acc)
    if "col_scale" in t:
        post = post * t["col_scale"].double()[None, :]
    if "rgs" in t:
        post = post * t["rgs"].double().repeat_interleave(c.rpg)[:c.M, None]
    if keep is not None:
        p = float(np.float32(c.drop))
        post = post * keep.to(acc.device, torch.float64) / (1.0 - p)
    R = y * post
    if "res" in t:
        R = R + t["res"].double()
    if "C0" in t:
        R = R + t["C0"]
    return R, z, gain * post.abs(), act_err * post.abs()


def bound(c, t, P, R, z, gain, act_err):
    """|C - R| <= C_ACC (|A|.|B|) gain + act_err + fp32 epilogue roundings + bf16 output rounding.  The accumulator's error,
    split-K slices included, is C_ACC (|A|.|B|); the fp32 term allows eight epilogue roundings at the magnitude of any
    intermediate (z = acc + bias carried through the scales, the residual, the accumulated C)."""
    mag = z.abs() * gain
    if "res" in t:
        mag = mag + t["res"].double().abs()
    if "C0" in t:
        mag = mag + t["C0"].abs()
    e_out = 2.0 ** -8 if c.out == BF16 else 0.0
    return C_ACC * P * gain + act_err + 8 * U32 * mag + e_out * R.abs()


def _ratio(err, bnd):
    """err / bound per element; 0 where both are 0 (a dropped element without residual is exactly 0)."""
    return torch.where(bnd > 0, err / bnd.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))


@pytest.mark.parametrize("c", CASES, ids=CASE_IDS)
def test_gemm_case(lib, record, c):
    """One row of CASES against the fp64 reference: per-element bound, canaries, the dropout mask, and two checks that the
    bound has teeth (a product missing one k-block and a slightly wrong reference both fail it)."""
    t = launch(lib, c, seed=1 + CASE_IDS.index(c.id))
    torch.cuda.synchronize()
    out = t["out"]
    assert out.outside_unchanged(), "C written outside [M, N]"
    if c.aux_out:
        assert t["aux_out"].outside_unchanged(), "aux_out written outside [M, N]"
    A, B = t["A"].double(), t["B"].double()
    acc, P = A @ B.t(), A.abs() @ B.abs().t()
    keep = keep_mask(c.M, c.N, 1 + CASE_IDS.index(c.id), c.drop).cuda() if c.drop else None
    R, z, gain, act_err = epilogue64(acc, t, c, keep)
    C = out.view.double()
    err = (C - R).abs()
    bnd = bound(c, t, P, R, z, gain, act_err)
    scaled = P * gain
    rest = bnd - C_ACC * scaled
    c_needed = float(((err - rest) / scaled.clamp_min(1e-300)).max())   # smallest C_ACC this case would pass
    worst = float(_ratio(err, bnd).max())
    if c.drop:   # the kept set is exactly the hash's: a dropped element is the residual / accumulated value, bit for bit
        base = torch.zeros_like(out.view)
        if "res" in t:
            base = base + t["res"].to(c.out)
        if "C0" in t:
            base = base + t["C0"].to(c.out)
        kept_by_kernel = out.view != base
    # the bound must not be loose enough to pass a product missing one 64-wide k-block
    frac = None
    if c.K >= 128:
        R_rm, _, _, _ = epilogue64(acc - A[:, :64] @ B[:, :64].t(), t, c, keep)
        sel = keep if keep is not None else torch.ones_like(R, dtype=torch.bool)
        frac = float((bnd < (R - R_rm).abs())[sel].double().mean())
    # a reference off by 2^-10 (f32) / 2^-6 (bf16) relative must fail
    rel = 2.0 ** -10 if c.out == F32 else 2.0 ** -6
    caught = bool(((C - R * (1 + rel)).abs() > bnd).any())
    aux_worst = None
    if c.aux_out:
        za = t["aux_out"].view.double()
        aux_worst = float(_ratio((za - z).abs(), C_ACC * P + (2.0 ** -8 + 8 * U32) * z.abs()).max())
    record("gemm_case", case=c.id, family=c.family, worst_ratio=worst, c_needed=c_needed, meaningful_frac=frac,
           aux_worst_ratio=aux_worst, perturbation_caught=caught)
    assert worst <= 1.0, (worst, c_needed)
    if aux_worst is not None:
        assert aux_worst <= 1.0, aux_worst
    if c.drop:
        assert torch.equal(kept_by_kernel, keep), "dropout kept set differs from drop_keep_idx"
    if frac is not None:
        assert frac >= 0.9, frac
    assert caught


def test_every_instantiation_is_reached(lib):
    """Each row of CASES runs the instantiation it names, and together they run all 24."""
    import re

    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i, c in enumerate(CASES):
            launch(lib, c, seed=1 + i)
        torch.cuda.synchronize()
    pat = re.compile(r"gemm_tcgen05_(pair_)?kernel<\s*(?:\(int\))?(\d+)\s*,\s*(?:\(int\))?(\d+)\s*,\s*(?:\(int\))?(\d+)\s*>")
    kern = [e for e in prof.events() if str(e.device_type).endswith("CUDA") and pat.search(e.name)]
    kern.sort(key=lambda e: e.time_range.start)
    seen = []
    for e in kern:
        m = pat.search(e.name)
        seen.append(("pair" if m.group(1) else "single") + "<%s,%s,%s>" % m.group(2, 3, 4))
    assert seen == [c.kernel for c in CASES], list(zip(CASE_IDS, seen))
    assert len(set(seen)) == 24


def test_split_k_linear_epilogue_matches_unsplit(lib):
    """col_scale, row_group_scale and dropout are linear in the accumulator with one mask for every K slice: split-K 3
    (one slice empty) and split-K 1 give the same result within the bound."""
    c = Case("split_linear", "epilogue", "pair<1,1,0>", "split-K with scales and dropout", 512, 512, 256, a_t=True,
             b_t=True, out=F32, acc=True, col_scale=True, rpg=17, drop=0.1)
    outs = []
    for split in (1, 3):
        t = launch(lib, c, seed=99, split=split)
        outs.append(t["out"].view.double())
    A, B = t["A"].double(), t["B"].double()
    keep = keep_mask(c.M, c.N, 99, c.drop).cuda()
    R, z, gain, act_err = epilogue64(A @ B.t(), t, c, keep)
    bnd = bound(c, t, A.abs() @ B.abs().t(), R, z, gain, act_err)
    assert bool(((outs[1] - outs[0]).abs() <= 2 * bnd).all())
    assert torch.equal(outs[1] == t["C0"], outs[0] == t["C0"])


# ------------------------------------------------------------------------------------------------ rejected arguments
REJECT = {
    "accumulate_bf16_out": dict(out=BF16, accumulate=True),
    "split_k_without_accumulate": dict(split_k=2),
    "dgelu_without_aux_in": dict(act=2, out=BF16),
    "misaligned_A": dict(a_off=1),
    "invalid_block_n": dict(block_n=96),
    "split_k_with_bias": dict(split_k=2, accumulate=True, bias=True),
    "split_k_with_residual": dict(split_k=2, accumulate=True, residual=True),
    "split_k_with_aux_out": dict(split_k=2, accumulate=True, aux_out=True),
    "split_k_with_gelu": dict(split_k=2, accumulate=True, act=1),
    "split_k_with_dgelu": dict(split_k=2, accumulate=True, act=2, aux_in=True),
    "split_k_with_tanh": dict(split_k=2, accumulate=True, act=3),
}


@pytest.mark.parametrize("name", list(REJECT))
def test_gemm_rejects(lib, name):
    """Host-side argument checks: RuntimeError before any launch, C untouched."""
    o = dict(REJECT[name])
    M, N, K = 256, 256, 256
    g = torch.Generator(device="cuda").manual_seed(5)
    a_off = o.pop("a_off", 0)
    abuf = torch.randn(M * K + a_off, device="cuda", generator=g).bfloat16()
    a = abuf[a_off:].view(M, K)
    b = torch.randn(N, K, device="cuda", generator=g).bfloat16()
    out = Buf(M, N, N + 8, o.pop("out", F32))
    if out.buf.dtype == F32:
        out.view.copy_(torch.randn(M, N, device="cuda", generator=g))
    kw = {}
    if o.pop("bias", False):
        kw["bias"] = torch.randn(N, device="cuda", generator=g)
    if o.pop("residual", False):
        kw["residual"] = torch.randn(M, N, device="cuda", generator=g)
    if o.pop("aux_out", False):
        kw["aux_out"] = torch.empty(M, N, dtype=BF16, device="cuda")
    if o.pop("aux_in", False):
        kw["aux_in"] = torch.randn(M, N, device="cuda", generator=g).bfloat16()
    kw.update(o)
    torch.cuda.synchronize()
    out.snapshot()
    with pytest.raises(RuntimeError):
        lib.gemm(a, b, out=out.view, **kw)
    torch.cuda.synchronize()
    assert out.unchanged()


# ------------------------------------------------------------------------------------------------ xfm_sgemm_f32
def _gamma(n):
    return n * U32 / (1 - n * U32)


def check_sgemm(L, A, B, out_buf, bias=None, accumulate=False):
    """One call of sgemm_f32 (A [M,K], B [N,K] views as given) against fp64.  The kernel is one fp32 FMA chain per element
    followed by the bias and accumulate adds: K + 2 roundings of partial sums bounded by |A|.|B| + |bias| + |C|."""
    C0 = out_buf.view.double().clone() if accumulate else None
    out_buf.snapshot()
    L.sgemm_f32(A, B, out=out_buf.view, bias=bias, accumulate=accumulate)
    Ad, Bd = A.double(), B.double()
    acc, mag = Ad @ Bd.t(), Ad.abs() @ Bd.abs().t()
    R = acc
    if bias is not None:
        R, mag = R + bias.double(), mag + bias.double().abs()
    if accumulate:
        R, mag = R + C0, mag + C0.abs()
    bnd = _gamma(A.shape[1] + 2) * mag
    C = out_buf.view.double()
    assert out_buf.outside_unchanged()
    err = (C - R).abs()
    assert bool((err <= bnd).all()), float((err / bnd).max())
    assert bool(((C - R * (1 + 2.0 ** -10)).abs() > bnd).any())
    if A.shape[1] >= 128:
        frac = float((bnd < (Ad[:, :64] @ Bd[:, :64].t()).abs()).double().mean())
        assert frac >= 0.9, frac
    return float((err / bnd).max())


SG_SIZES = (1, 31, 32, 33, 257)


@pytest.mark.parametrize("ta,tb", list(itertools.product((False, True), repeat=2)))
def test_sgemm_f32_shapes(lib, record, ta, tb):
    """Every transpose combination (passed as .t() views) over M, N, K in {1, 31, 32, 33, 257}; bias, accumulate and ldc > N
    on alternating shapes."""
    g = torch.Generator(device="cuda").manual_seed(7 + 2 * ta + tb)
    worst = 0.0
    for i, (M, N, K) in enumerate(itertools.product(SG_SIZES, repeat=3)):
        A = torch.randn(K, M, device="cuda", generator=g).t() if ta else torch.randn(M, K, device="cuda", generator=g)
        B = torch.randn(K, N, device="cuda", generator=g).t() if tb else torch.randn(N, K, device="cuda", generator=g)
        bias = torch.randn(N, device="cuda", generator=g) if i % 2 else None
        out = Buf(M, N, N + (3 if i % 3 else 0), F32)
        acc = i % 4 == 1
        if acc:
            out.view.copy_(torch.randn(M, N, device="cuda", generator=g))
        worst = max(worst, check_sgemm(lib, A, B, out, bias=bias, accumulate=acc))
    record("sgemm_shapes", ta=ta, tb=tb, worst_ratio=worst)


def test_sgemm_f32_model_calls(lib, record):
    """The calls of encoders.ProjHead (B = 96, D = 768, E = 256, CLS rows with row stride Lt * D) and one retrieval-sized
    similarity product (1000 x 256 against 5000 x 256)."""
    g = torch.Generator(device="cuda").manual_seed(11)
    Bn, Lt, D, E = 96, 40, 768, 256
    emb = torch.randn(Bn, Lt * D, device="cuda", generator=g)
    x0 = emb[:, :D]
    W = torch.randn(E, D, device="cuda", generator=g) * D ** -0.5
    bias = torch.randn(E, device="cuda", generator=g)
    dz = torch.randn(Bn, E, device="cuda", generator=g)
    ones = torch.ones((1, Bn), device="cuda")
    worst = []
    worst.append(check_sgemm(lib, x0, W, Buf(Bn, E, E, F32), bias=bias))                      # z = x0 W^T + b
    db = Buf(E, 1, 1, F32)
    db.view.copy_(torch.randn(E, 1, device="cuda", generator=g))
    worst.append(check_sgemm(lib, dz.t(), ones, db, accumulate=True))                         # db += dz^T 1
    dW = Buf(E, D, D, F32)
    dW.view.copy_(torch.randn(E, D, device="cuda", generator=g))
    worst.append(check_sgemm(lib, dz.t(), x0.t(), dW, accumulate=True))                       # dW += dz^T x0
    worst.append(check_sgemm(lib, dz, W.t(), Buf(Bn, D, Lt * D, F32)))                         # dx0 = dz W
    img = torch.nn.functional.normalize(torch.randn(1000, E, device="cuda", generator=g), dim=-1)
    txt = torch.nn.functional.normalize(torch.randn(5000, E, device="cuda", generator=g), dim=-1)
    worst.append(check_sgemm(lib, img, txt, Buf(1000, 5000, 5000, F32)))                      # retrieval similarities
    record("sgemm_model_calls", worst_ratio=max(worst))
