"""ctypes binding of libxfm_b200.so (the C-ABI declared in include/xfm_b200.h).

The library is the only compute path of this package: there is no CPU or eager-PyTorch
fallback.  If the shared object is missing, or a GPU is required and absent, calls raise.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxfm_b200.so")

_lib = None
_inited_devices = set()
gemm_profile = None  # set to a list to time every GEMM launch with CUDA events (bench.py)
# block_n = 0 (auto) picks the CTA-pair (cta_group::2, 256 x 256 tiles) kernel for problems with at least this many rows
PAIR_MIN_M = int(os.environ.get("XFM_GEMM_PAIR_MIN_M", "2048"))


class GemmParams(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("B", C.c_void_p), ("C", C.c_void_p),
        ("lda", C.c_int64), ("ldb", C.c_int64), ("ldc", C.c_int64),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("a_mn_major", C.c_int32), ("b_mn_major", C.c_int32),
        ("c_dtype", C.c_int32), ("split_k", C.c_int32), ("accumulate", C.c_int32),
        ("act", C.c_int32), ("res_dtype", C.c_int32), ("rows_per_group", C.c_int32),
        ("block_n", C.c_int32),
        ("bias", C.c_void_p), ("aux_in", C.c_void_p), ("aux_out", C.c_void_p),
        ("ld_aux_in", C.c_int64), ("ld_aux_out", C.c_int64), ("ld_res", C.c_int64),
        ("col_scale", C.c_void_p), ("row_group_scale", C.c_void_p), ("residual", C.c_void_p),
        ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64),
    ]


def load():
    """Load the shared library (no CUDA context needed).  Raises if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(xfm_b200 has no fallback path)")
        _lib = C.CDLL(LIB_PATH)
        _lib.xfm_version.restype = C.c_int
        _lib.xfm_init.restype = C.c_int
        _lib.xfm_launch_count.restype = C.c_int64
        _lib.xfm_last_error.restype = C.c_char_p
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().xfm_last_error().decode()
        raise RuntimeError(f"xfm_b200: {what} failed with code {rc}: {msg}")


_cur_dev = torch._C._cuda_getDevice if hasattr(torch._C, "_cuda_getDevice") else None
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def lib():
    """Library handle, initialised for the current CUDA device (hot path: one C call + a set lookup)."""
    if _lib is not None and _inited_devices:
        dev = _cur_dev() if _cur_dev is not None else torch.cuda.current_device()
        if dev in _inited_devices:
            return _lib
    l = load()
    if not torch.cuda.is_available():
        raise RuntimeError("xfm_b200 needs a CUDA device (sm_100a); there is no CPU path")
    dev = torch.cuda.current_device()
    if dev not in _inited_devices:
        torch.cuda.init()
        torch.zeros(1, device="cuda")  # make sure the primary context exists
        check(l.xfm_init(), "xfm_init")
        _inited_devices.add(dev)
    return l


def seed_salt_bump(inc=1):
    """Advance the device-resident word every dropout / sampling kernel adds to its seed (capturable: one tiny kernel)."""
    check(lib().xfm_seed_salt_bump(C.c_uint64(inc), stream_ptr()), "xfm_seed_salt_bump")


def seed_salt_set(value=0):
    check(lib().xfm_seed_salt_set(C.c_uint64(value), stream_ptr()), "xfm_seed_salt_set")


def launch_count():
    return int(load().xfm_launch_count())


def stream_ptr():
    """Raw cudaStream_t of torch's current stream on the current device."""
    if _raw_stream is not None and _cur_dev is not None:
        return C.c_void_p(_raw_stream(_cur_dev()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


_DT = {torch.bfloat16: 0, torch.float32: 1}


def gemm(a, b, *, a_t=False, b_t=False, out=None, out_dtype=torch.bfloat16, bias=None, act=0, aux_in=None,
         aux_out=None, col_scale=None, row_group_scale=None, rows_per_group=1, residual=None, dropout_p=0.0,
         dropout_seed=0, accumulate=False, split_k=1, block_n=0):
    """C[M,N] = epilogue(A · B^T).

    a: bf16 [M,K] (or [K,M] with a_t=True: the stored tensor is the transpose, "MN-major").
    b: bf16 [N,K] (or [K,N] with b_t=True).
    split_k > 1 needs an f32 `out` with accumulate=True and rejects bias, residual, aux_out and act != 0: every K slice
    applies the epilogue to its partial sum, so only col_scale, row_group_scale and dropout may be combined with it.
    """
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    assert a.dim() == 2 and b.dim() == 2 and a.stride(1) == 1 and b.stride(1) == 1
    if a_t:
        K, M = a.shape
    else:
        M, K = a.shape
    if b_t:
        Kb, N = b.shape
    else:
        N, Kb = b.shape
    assert K == Kb, (a.shape, b.shape, a_t, b_t)
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    assert out.shape == (M, N) and out.stride(1) == 1
    p = GemmParams()
    p.A, p.B, p.C = a.data_ptr(), b.data_ptr(), out.data_ptr()
    p.lda, p.ldb, p.ldc = a.stride(0), b.stride(0), out.stride(0)
    p.M, p.N, p.K = M, N, K
    p.a_mn_major, p.b_mn_major = int(a_t), int(b_t)
    p.c_dtype = _DT[out.dtype]
    p.split_k = split_k
    p.accumulate = int(accumulate)
    p.act = act
    if block_n == 0 and M >= PAIR_MIN_M and N >= 256:
        block_n = 512
    p.block_n = block_n
    p.rows_per_group = rows_per_group
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N
        p.bias = bias.data_ptr()
    if aux_in is not None:
        assert aux_in.dtype == torch.bfloat16 and aux_in.shape == (M, N)
        p.aux_in, p.ld_aux_in = aux_in.data_ptr(), aux_in.stride(0)
    if aux_out is not None:
        assert aux_out.dtype == torch.bfloat16 and aux_out.shape == (M, N)
        p.aux_out, p.ld_aux_out = aux_out.data_ptr(), aux_out.stride(0)
    if col_scale is not None:
        assert col_scale.dtype == torch.float32 and col_scale.numel() == N
        p.col_scale = col_scale.data_ptr()
    if row_group_scale is not None:
        assert row_group_scale.dtype == torch.float32
        p.row_group_scale = row_group_scale.data_ptr()
    if residual is not None:
        assert residual.shape == (M, N) and residual.stride(1) == 1
        p.residual, p.ld_res, p.res_dtype = residual.data_ptr(), residual.stride(0), _DT[residual.dtype]
    p.dropout_p = dropout_p
    p.dropout_seed = dropout_seed
    if gemm_profile is not None:  # bench.py roofline leg: CUDA events around every launch of the dominant kernel
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib().xfm_gemm_bf16(C.byref(p), stream_ptr()), "xfm_gemm_bf16")
        e1.record()
        # algorithmic bytes of this launch: both operands once, the output once (read too when accumulating), every
        # epilogue operand once
        nbytes = 2 * (M * K + N * K) + out.element_size() * M * N * (2 if accumulate else 1)
        for t in (aux_in, aux_out, residual):
            if t is not None:
                nbytes += t.element_size() * M * N
        gemm_profile.append((2.0 * M * N * K, e0, e1, (M, N, K, int(a_t), int(b_t)), nbytes))
        return out
    check(lib().xfm_gemm_bf16(C.byref(p), stream_ptr()), "xfm_gemm_bf16")
    return out


# ------------------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------------------
class AttnParams(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p), ("lse", C.c_void_p),
        ("bias", C.c_void_p), ("kmask", C.c_void_p), ("kv_index", C.c_void_p),
        ("q_stride", C.c_int64), ("k_stride", C.c_int64), ("v_stride", C.c_int64), ("o_stride", C.c_int64),
        ("bias_ld", C.c_int64),
        ("B", C.c_int32), ("H", C.c_int32), ("Lq", C.c_int32), ("Lk", C.c_int32), ("head_dim", C.c_int32),
        ("Bkv", C.c_int32),
        ("scale", C.c_float), ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64),
        ("dout", C.c_void_p), ("delta", C.c_void_p),
        ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p), ("ds_dump", C.c_void_p),
        ("do_stride", C.c_int64), ("dq_stride", C.c_int64), ("dk_stride", C.c_int64), ("dv_stride", C.c_int64),
        ("ds_ld", C.c_int64),
        ("kv_offsets", C.c_void_p), ("kv_samples", C.c_void_p),
        ("rel_table", C.c_void_p), ("rel_window", C.c_int32), ("allow_tc", C.c_int32),
        ("part_out", C.c_void_p), ("part_lse", C.c_void_p),
    ]


def _attn_common(p, q, k, v, B, H, Lq, Lk, Bkv, scale, bias, kmask, kv_index, dropout_p, dropout_seed):
    for t in (q, k, v):
        assert t.dtype == torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1
    assert q.shape[0] == B * Lq and k.shape[0] == Bkv * Lk and v.shape[0] == Bkv * Lk
    p.q, p.k, p.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    p.q_stride, p.k_stride, p.v_stride = q.stride(0), k.stride(0), v.stride(0)
    p.B, p.H, p.Lq, p.Lk, p.head_dim, p.Bkv = B, H, Lq, Lk, 64, Bkv
    p.scale, p.dropout_p, p.dropout_seed = scale, dropout_p, dropout_seed
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.dim() == 3 and bias.shape[0] == H and bias.shape[1] == Lq
        assert bias.stride(2) == 1 and bias.stride(0) == Lq * bias.stride(1)
        p.bias, p.bias_ld = bias.data_ptr(), bias.stride(1)
    if kmask is not None:
        assert kmask.dtype == torch.float32 and kmask.shape == (B, Lk) and kmask.is_contiguous()
        p.kmask = kmask.data_ptr()
    if kv_index is not None:
        assert kv_index.dtype == torch.int32 and kv_index.numel() == B
        p.kv_index = kv_index.data_ptr()


def attention_fwd(q, k, v, B, H, Lq, Lk, scale, *, Bkv=None, bias=None, kmask=None, kv_index=None, dropout_p=0.0,
                  dropout_seed=0, out=None, rel_table=None, rel_window=0, allow_tc=True, kv_offsets=None, kv_samples=None):
    """q: bf16 [B*Lq, >=H*64] view; k, v: bf16 [Bkv*Lk, ...] views.  Returns (out bf16 [B*Lq, H*64], lse f32 [B,H,Lq]).
    rel_table / rel_window: BEiT relative-position table [(2W-1)^2+3, H] f32 whose closed-form gather equals `bias`
    (tcgen05 path); allow_tc=False forces the mma.sync kernel."""
    Bkv = B if Bkv is None else Bkv
    if out is None:
        out = torch.empty((B * Lq, H * 64), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((B, H, Lq), dtype=torch.float32, device=q.device)
    p = AttnParams()
    _attn_common(p, q, k, v, B, H, Lq, Lk, Bkv, scale, bias, kmask, kv_index, dropout_p, dropout_seed)
    p.out, p.o_stride, p.lse = out.data_ptr(), out.stride(0), lse.data_ptr()
    p.allow_tc = int(allow_tc)
    if rel_table is not None:
        assert rel_table.dtype == torch.float32 and rel_table.is_contiguous() and rel_table.shape[1] == H
        assert rel_table.shape[0] == (2 * rel_window - 1) ** 2 + 3
        p.rel_table, p.rel_window = rel_table.data_ptr(), rel_window
    if kv_samples is not None:  # CSR inverse of kv_index: lets the tcgen05 cross-attention kernel stack the samples of an image
        assert kv_offsets.dtype == torch.int32 and kv_samples.dtype == torch.int32
        assert kv_offsets.numel() == Bkv + 1 and kv_samples.numel() == B
        p.kv_offsets, p.kv_samples = kv_offsets.data_ptr(), kv_samples.data_ptr()
    nb = load().xfm_attention_fwd_parts(C.byref(p))
    if nb:  # tcgen05 path in key blocks (384 / 480 px): one launch per block + a merge; scratch for the partial results
        parts = (torch.empty((nb, B * Lq, H * 64), dtype=torch.bfloat16, device=q.device),
                 torch.empty((nb, B, H, Lq), dtype=torch.float32, device=q.device))
        p.part_out, p.part_lse = parts[0].data_ptr(), parts[1].data_ptr()
    check(lib().xfm_attention_fwd(C.byref(p), stream_ptr()), "xfm_attention_fwd")
    return out, lse


def attention_bwd(dout, q, k, v, out, lse, B, H, Lq, Lk, scale, dq, dk, dv, *, Bkv=None, bias=None, kmask=None,
                  kv_index=None, kv_offsets=None, kv_samples=None, dropout_p=0.0, dropout_seed=0, ds_dump=None,
                  rel_table=None, rel_window=0, allow_tc=True):
    """Writes bf16 dq [B*Lq, ...], dk / dv [Bkv*Lk, ...] (views with row strides).  ds_dump: bf16 [B,H,Lq,ld] receives dS;
    the caller reduces it into the bias-table gradient (batch_sum_bf16, relpos_bias_bwd).  rel_table / rel_window:
    closed-form relative-position bias [(2W-1)^2+3, H] f32 whose gather equals `bias` (tcgen05 path)."""
    Bkv = B if Bkv is None else Bkv
    p = AttnParams()
    _attn_common(p, q, k, v, B, H, Lq, Lk, Bkv, scale, bias, kmask, kv_index, dropout_p, dropout_seed)
    delta = torch.empty((B, H, Lq), dtype=torch.float32, device=q.device)
    assert dout.dtype == torch.bfloat16 and dout.stride(1) == 1 and out.stride(1) == 1
    p.out, p.o_stride, p.lse = out.data_ptr(), out.stride(0), lse.data_ptr()
    p.dout, p.do_stride, p.delta = dout.data_ptr(), dout.stride(0), delta.data_ptr()
    for t in (dq, dk, dv):
        assert t.dtype == torch.bfloat16 and t.stride(1) == 1
    p.dq, p.dk, p.dv = dq.data_ptr(), dk.data_ptr(), dv.data_ptr()
    p.dq_stride, p.dk_stride, p.dv_stride = dq.stride(0), dk.stride(0), dv.stride(0)
    if ds_dump is not None:
        assert ds_dump.dtype == torch.bfloat16 and ds_dump.is_contiguous() and ds_dump.shape[:3] == (B, H, Lq)
        p.ds_dump, p.ds_ld = ds_dump.data_ptr(), ds_dump.shape[3]
    if kv_samples is not None:
        assert kv_offsets.dtype == torch.int32 and kv_samples.dtype == torch.int32
        p.kv_offsets, p.kv_samples = kv_offsets.data_ptr(), kv_samples.data_ptr()
    p.allow_tc = int(allow_tc)
    if rel_table is not None:
        assert rel_table.dtype == torch.float32 and rel_table.is_contiguous() and rel_table.shape[1] == H
        assert rel_table.shape[0] == (2 * rel_window - 1) ** 2 + 3
        p.rel_table, p.rel_window = rel_table.data_ptr(), rel_window
    check(lib().xfm_attention_bwd(C.byref(p), stream_ptr()), "xfm_attention_bwd")


class VarlenParams(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p), ("lse", C.c_void_p),
        ("q_stride", C.c_int64), ("k_stride", C.c_int64), ("v_stride", C.c_int64), ("o_stride", C.c_int64),
        ("cu_seqlens", C.c_void_p), ("tiles", C.c_void_p),
        ("n", C.c_int32), ("n_tiles", C.c_int32), ("H", C.c_int32), ("Lpad", C.c_int32), ("T", C.c_int32),
        ("scale", C.c_float), ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64),
        ("dout", C.c_void_p), ("delta", C.c_void_p),
        ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p),
        ("do_stride", C.c_int64), ("dq_stride", C.c_int64), ("dk_stride", C.c_int64), ("dv_stride", C.c_int64),
    ]


def varlen_plan(lengths):
    """Sequence lengths (1..128 each) -> (cu_seqlens int32 [n+1], tiles int32 [n_tiles+1]) on the host: the packed row
    offsets and the tiles of xfm_attention_varlen_plan (first sequence of every tile, then n).  Needs no device."""
    ln = torch.as_tensor(lengths, dtype=torch.int32).reshape(-1).contiguous()
    n = ln.numel()
    cu = torch.empty(n + 1, dtype=torch.int32)
    tiles = torch.empty(n + 1, dtype=torch.int32)
    nt = C.c_int32(0)
    check(load().xfm_attention_varlen_plan(C.c_void_p(ln.data_ptr()), n, C.c_void_p(cu.data_ptr()),
                                           C.c_void_p(tiles.data_ptr()), C.byref(nt)), "xfm_attention_varlen_plan")
    return cu, tiles[:nt.value + 1].clone()


def _varlen_common(p, q, k, v, cu_seqlens, tiles, H, Lpad, scale, dropout_p, dropout_seed):
    for t in (q, k, v):
        assert t.dtype == torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1 and t.shape[1] == H * 64
    assert q.shape[0] == k.shape[0] == v.shape[0]
    for t in (cu_seqlens, tiles):
        assert t.dtype == torch.int32 and t.is_contiguous() and t.device == q.device
    p.q, p.k, p.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    p.q_stride, p.k_stride, p.v_stride = q.stride(0), k.stride(0), v.stride(0)
    p.cu_seqlens, p.tiles = cu_seqlens.data_ptr(), tiles.data_ptr()
    p.n, p.n_tiles, p.H, p.Lpad, p.T = cu_seqlens.numel() - 1, tiles.numel() - 1, H, Lpad, q.shape[0]
    p.scale, p.dropout_p, p.dropout_seed = scale, dropout_p, dropout_seed


def attention_varlen_fwd(q, k, v, cu_seqlens, tiles, H, Lpad, scale, *, dropout_p=0.0, dropout_seed=0, out=None):
    """Packed variable-length self-attention.  q, k, v: bf16 [T, H*64] views (row strides allowed); cu_seqlens / tiles:
    int32 device copies of varlen_plan's output; Lpad: the padded length the batch arrived in (numbers the dropout mask as
    the padded layout does).  Returns (out bf16 [T, H*64], lse f32 [H, T])."""
    T = q.shape[0]
    if out is None:
        out = torch.empty((T, H * 64), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((H, T), dtype=torch.float32, device=q.device)
    p = VarlenParams()
    _varlen_common(p, q, k, v, cu_seqlens, tiles, H, Lpad, scale, dropout_p, dropout_seed)
    assert out.shape == (T, H * 64) and out.stride(1) == 1
    p.out, p.o_stride, p.lse = out.data_ptr(), out.stride(0), lse.data_ptr()
    check(lib().xfm_attention_varlen_fwd(C.byref(p), stream_ptr()), "xfm_attention_varlen_fwd")
    return out, lse


def attention_varlen_bwd(dout, q, k, v, out, lse, cu_seqlens, tiles, H, Lpad, scale, dq, dk, dv, *, dropout_p=0.0,
                         dropout_seed=0):
    """Writes bf16 dq / dk / dv [T, H*64] (views with row strides) of attention_varlen_fwd."""
    p = VarlenParams()
    _varlen_common(p, q, k, v, cu_seqlens, tiles, H, Lpad, scale, dropout_p, dropout_seed)
    T = q.shape[0]
    assert lse.shape == (H, T) and lse.dtype == torch.float32 and lse.is_contiguous()
    delta = torch.empty((H, T), dtype=torch.float32, device=q.device)
    for t in (dout, out, dq, dk, dv):
        assert t.dtype == torch.bfloat16 and t.stride(1) == 1 and t.shape == (T, H * 64)
    p.out, p.o_stride, p.lse = out.data_ptr(), out.stride(0), lse.data_ptr()
    p.dout, p.do_stride, p.delta = dout.data_ptr(), dout.stride(0), delta.data_ptr()
    p.dq, p.dk, p.dv = dq.data_ptr(), dk.data_ptr(), dv.data_ptr()
    p.dq_stride, p.dk_stride, p.dv_stride = dq.stride(0), dk.stride(0), dv.stride(0)
    check(lib().xfm_attention_varlen_bwd(C.byref(p), stream_ptr()), "xfm_attention_varlen_bwd")


def vit_attention_bwd_tc_ok(n_tokens):
    """Token counts the fused tcgen05 backward handles: the forward's plus 577 (384 px) and 901 (480 px), processed in key
    blocks of about 192 keys (three and five)."""
    return n_tokens in (197, 145, 50, 17, 577, 901)


# ------------------------------------------------------------------------------------------------------
# thin wrappers over the remaining entry points
# ------------------------------------------------------------------------------------------------------
def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _dt(t):
    return _DT[t.dtype]


def layernorm_fwd(x, w, b, eps, out_dtype=torch.bfloat16, want_f32_copy=False, want_stats=True):
    M, D = x.shape
    assert x.is_contiguous()
    y = torch.empty((M, D), dtype=out_dtype, device=x.device)
    y2 = torch.empty((M, D), dtype=torch.float32, device=x.device) if want_f32_copy else None
    stats = torch.empty((M, 2), dtype=torch.float32, device=x.device) if want_stats else None
    check(lib().xfm_layernorm_fwd(_p(x), _dt(x), _p(w), _p(b), _p(y), _dt(y), _p(y2), _p(stats), M, D, C.c_float(eps),
                                  stream_ptr()), "xfm_layernorm_fwd")
    return y, stats, y2


def layernorm_bwd(dy, x, stats, w, dw, db, add_in=None, out_dtype=torch.float32):
    M, D = x.shape
    assert dy.is_contiguous() and x.is_contiguous() and dy.shape == x.shape
    dx = torch.empty((M, D), dtype=out_dtype, device=x.device)
    check(lib().xfm_layernorm_bwd(_p(dy), _dt(dy), _p(x), _dt(x), _p(stats), _p(w), _p(add_in),
                                  0 if add_in is None else _dt(add_in), _p(dx), _dt(dx), _p(dw), _p(db), M, D,
                                  stream_ptr()), "xfm_layernorm_bwd")
    return dx


def layernorm_bwd_dense(dy, x, stats, w, dw, db, dbias, drop_p=0.0, drop_seed=0, out_dtype=torch.float32):
    """LayerNorm backward that also returns dx16 = bf16(dropout_mask * dx / (1 - p)) and accumulates its column sums into
    `dbias` (see xfm_layernorm_bwd_dense).  Returns (dx, dx16)."""
    M, D = x.shape
    assert dy.is_contiguous() and x.is_contiguous() and dy.shape == x.shape and dbias.dtype == torch.float32
    dx = torch.empty((M, D), dtype=out_dtype, device=x.device)
    dx16 = torch.empty((M, D), dtype=torch.bfloat16, device=x.device)
    check(lib().xfm_layernorm_bwd_dense(_p(dy), _dt(dy), _p(x), _dt(x), _p(stats), _p(w), _p(None), 0, _p(dx), _dt(dx), _p(dw),
                                        _p(db), _p(dx16), _p(dbias), C.c_float(drop_p), C.c_uint64(drop_seed), M, D,
                                        stream_ptr()), "xfm_layernorm_bwd_dense")
    return dx, dx16


def layerscale_bwd(dx_out, z, gamma, dgamma, dbias, row_group_scale=None, rows_per_group=1):
    M, D = dx_out.shape
    assert dx_out.dtype == torch.float32 and z.dtype == torch.bfloat16 and dx_out.is_contiguous() and z.is_contiguous()
    dz = torch.empty((M, D), dtype=torch.bfloat16, device=z.device)
    check(lib().xfm_layerscale_bwd(_p(dx_out), _p(z), _p(gamma), _p(row_group_scale), rows_per_group, _p(dz), _p(dgamma),
                                   _p(dbias), M, D, stream_ptr()), "xfm_layerscale_bwd")
    return dz


def colsum_into(x, out):
    """out[c] += sum_rows x[:, c]; x bf16 2-D (row stride allowed)."""
    assert x.dtype == torch.bfloat16 and x.stride(1) == 1 and out.dtype == torch.float32
    check(lib().xfm_colsum_bf16(_p(x), C.c_int64(x.stride(0)), _p(out), x.shape[0], x.shape[1], stream_ptr()),
          "xfm_colsum_bf16")


def cast_to_bf16(src, dst):
    assert src.dtype == torch.float32 and dst.dtype == torch.bfloat16 and src.numel() == dst.numel()
    assert src.is_contiguous() and dst.is_contiguous()
    check(lib().xfm_cast_f32_to_bf16(_p(src), _p(dst), C.c_size_t(src.numel()), stream_ptr()), "xfm_cast_f32_to_bf16")


def cast_to_f32(src, dst):
    assert src.dtype == torch.bfloat16 and dst.dtype == torch.float32 and src.numel() == dst.numel()
    check(lib().xfm_cast_bf16_to_f32(_p(src), _p(dst), C.c_size_t(src.numel()), stream_ptr()), "xfm_cast_bf16_to_f32")


def split_bf16x3(x, role, act=0):
    """f32 [M, K] -> bf16 [M, 6K]: three-term bf16 split laid out for an fp32-grade GEMM over K' = 6K (role 0 = left operand,
    1 = right operand / weight; act=1 applies tanh first).  See xfm_split_bf16x3."""
    assert x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous()
    M, K = x.shape
    out = torch.empty((M, 6 * K), dtype=torch.bfloat16, device=x.device)
    check(lib().xfm_split_bf16x3(_p(x), _p(out), M, K, role, act, stream_ptr()), "xfm_split_bf16x3")
    return out


def scale_by_scalar(t, scalar):
    """t * scalar[0] as a NEW tensor (scalar: f32 [1] on the device)."""
    assert t.is_contiguous() and scalar.dtype == torch.float32
    out = torch.empty_like(t)
    check(lib().xfm_scale_by_scalar(_p(t), _p(out), _dt(t), _p(scalar), C.c_size_t(t.numel()), stream_ptr()), "xfm_scale_by_scalar")
    return out


def roberta_embed_fwd(ids, word, pos, type_emb, ln_w, ln_b, pad_id, eps, want_pre=True, absolute_pos=False):
    B, L = ids.shape
    D = word.shape[1]
    assert ids.dtype == torch.int64 and ids.is_contiguous()
    y = torch.empty((B * L, D), dtype=torch.bfloat16, device=ids.device)
    pre = torch.empty((B * L, D), dtype=torch.float32, device=ids.device) if want_pre else None
    stats = torch.empty((B * L, 2), dtype=torch.float32, device=ids.device)
    pos_ids = torch.empty((B, L), dtype=torch.int32, device=ids.device)
    check(lib().xfm_roberta_embed_fwd(_p(ids), _p(word), _p(pos), _p(type_emb), _p(ln_w), _p(ln_b), _p(y), _p(pre),
                                      _p(stats), _p(pos_ids), B, L, D, pad_id, int(absolute_pos), C.c_float(eps), stream_ptr()),
          "xfm_roberta_embed_fwd")
    return y, pre, stats, pos_ids


def roberta_embed_bwd(dpre, ids, pos_ids, dword, dpos, dtype0, word_pad, pos_pad=None):
    rows, D = dpre.shape
    pos_pad = word_pad if pos_pad is None else pos_pad
    check(lib().xfm_roberta_embed_bwd(_p(dpre), _p(ids), _p(pos_ids), _p(dword), _p(dpos), _p(dtype0), rows, D, word_pad,
                                      pos_pad, stream_ptr()), "xfm_roberta_embed_bwd")


def im2col(image, P, pre_mul=None):
    """pre_mul: None, or a 1-element f32 DEVICE tensor m: pixels become x * m / 127.5 - 1 (model_vqkd.py:125-131)."""
    B, Cc, H, W = image.shape
    assert image.dtype == torch.float32 and image.is_contiguous()
    assert pre_mul is None or (pre_mul.dtype == torch.float32 and pre_mul.is_cuda and pre_mul.numel() == 1)
    out = torch.empty((B * (H // P) * (W // P), Cc * P * P), dtype=torch.bfloat16, device=image.device)
    check(lib().xfm_im2col(_p(image), _p(out), B, Cc, H, W, P, _p(pre_mul), stream_ptr()), "xfm_im2col")
    return out


def assemble_tokens(patch, cls, mask_token, mask_u8, pos, B, npatch, out=None):
    D = patch.shape[1]
    x = out if out is not None else torch.empty((B * (npatch + 1), D), dtype=torch.float32, device=patch.device)
    assert x.shape == (B * (npatch + 1), D) and x.dtype == torch.float32 and x.is_contiguous()
    check(lib().xfm_assemble_tokens(_p(patch), _p(cls), _p(mask_token), _p(mask_u8), _p(pos), _p(x), B, npatch, D,
                                    stream_ptr()), "xfm_assemble_tokens")
    return x


def assemble_tokens_bwd(dx, mask_u8, dcls, dmask_token, B, npatch):
    D = dx.shape[1]
    dpatch = torch.empty((B * npatch, D), dtype=torch.bfloat16, device=dx.device)
    check(lib().xfm_assemble_tokens_bwd(_p(dx), _p(mask_u8), _p(dpatch), _p(dcls), _p(dmask_token), B, npatch, D,
                                        stream_ptr()), "xfm_assemble_tokens_bwd")
    return dpatch


def meanpool_fwd_(y_bf16, y_f32, B, npatch):
    check(lib().xfm_meanpool_fwd(_p(y_bf16), _p(y_f32), B, npatch, y_f32.shape[-1], stream_ptr()), "xfm_meanpool_fwd")


def meanpool_bwd(dout, B, npatch):
    dy = torch.empty_like(dout)
    check(lib().xfm_meanpool_bwd(_p(dout), _p(dy), B, npatch, dout.shape[-1], stream_ptr()), "xfm_meanpool_bwd")
    return dy


def gather_rows(src, index, out_dtype=None):
    assert src.dim() == 2 and src.is_contiguous() and index.dtype == torch.int64
    out = torch.empty((index.numel(), src.shape[1]), dtype=out_dtype or src.dtype, device=src.device)
    check(lib().xfm_gather_rows(_p(src), _dt(src), _p(index), _p(out), _dt(out), index.numel(), src.shape[1],
                                stream_ptr()), "xfm_gather_rows")
    return out


def scatter_add_rows_(dst, index, src):
    assert dst.dtype == torch.float32 and dst.is_contiguous() and src.is_contiguous() and index.dtype == torch.int64
    check(lib().xfm_scatter_add_rows(_p(src), _dt(src), _p(index), _p(dst), index.numel(), src.shape[1], stream_ptr()),
          "xfm_scatter_add_rows")


def relpos_bias_fwd(table, index, N, H, ld):
    bias = torch.zeros((H, N, ld), dtype=torch.float32, device=table.device)
    check(lib().xfm_relpos_bias_fwd(_p(table), _p(index), _p(bias), N, ld, H, stream_ptr()), "xfm_relpos_bias_fwd")
    return bias


def relpos_bias_bwd(dbias, index, dtable, N, H, ld):
    check(lib().xfm_relpos_bias_bwd(_p(dbias), _p(index), _p(dtable), N, ld, H, stream_ptr()), "xfm_relpos_bias_bwd")


def batch_sum_bf16(x):
    """x bf16 [B, ...] -> f32 [...] summed over dim 0."""
    B = x.shape[0]
    per = x[0].numel()
    out = torch.empty(x.shape[1:], dtype=torch.float32, device=x.device)
    check(lib().xfm_batch_sum_bf16(_p(x), _p(out), B, C.c_size_t(per), stream_ptr()), "xfm_batch_sum_bf16")
    return out


def ce_fwd(logits, labels, V, want_rows=False):
    """logits f32 [R, ld>=V]; labels int64 [R] (-100 = ignore).  Returns (loss[1], count[1], lse[R]) and, with want_rows,
    the per-row losses [R] (0 for ignored rows) as a fourth value."""
    R = logits.shape[0]
    assert logits.dtype == torch.float32 and logits.stride(1) == 1 and labels.dtype == torch.int64
    dev = logits.device
    row_loss = torch.empty(R, dtype=torch.float32, device=dev)
    lse = torch.empty(R, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    count = torch.empty(1, dtype=torch.float32, device=dev)
    check(lib().xfm_ce_fwd(_p(logits), C.c_int64(logits.stride(0)), _p(labels), R, V, _p(row_loss), _p(lse), _p(loss),
                           _p(count), stream_ptr()), "xfm_ce_fwd")
    if want_rows:
        return loss, count, lse, row_loss
    return loss, count, lse


def ce_bwd(logits, labels, lse, count, upstream, V, ldd):
    R = logits.shape[0]
    d = torch.empty((R, ldd), dtype=torch.bfloat16, device=logits.device)
    check(lib().xfm_ce_bwd(_p(logits), C.c_int64(logits.stride(0)), _p(labels), _p(lse), _p(count), _p(upstream), _p(d),
                           C.c_int64(ldd), R, V, stream_ptr()), "xfm_ce_bwd")
    return d


def ce_bwd_rows(logits, labels, lse, row_scale, upstream, V, ldd):
    """dlogits bf16 [R, ldd] = (softmax - onehot) * row_scale[row] * upstream (reduction='none' + weighted sum)."""
    R = logits.shape[0]
    assert row_scale.dtype == torch.float32 and row_scale.numel() == R and row_scale.is_contiguous()
    d = torch.empty((R, ldd), dtype=torch.bfloat16, device=logits.device)
    check(lib().xfm_ce_bwd_rows(_p(logits), C.c_int64(logits.stride(0)), _p(labels), _p(lse), _p(row_scale), _p(upstream),
                                _p(d), C.c_int64(ldd), R, V, stream_ptr()), "xfm_ce_bwd_rows")
    return d


def itc_loss_fused(image_all, text_all, temp, local_off, local_n, idx_all=None):
    n, E = image_all.shape
    dev = image_all.device
    l = lib()
    l.xfm_itc_workspace.restype = C.c_size_t
    work = torch.empty(l.xfm_itc_workspace(n), dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    dtemp = torch.empty(1, dtype=torch.float32, device=dev)
    di = torch.empty((local_n, E), dtype=torch.float32, device=dev)
    dt = torch.empty((local_n, E), dtype=torch.float32, device=dev)
    assert image_all.is_contiguous() and text_all.is_contiguous() and image_all.dtype == torch.float32
    check(l.xfm_itc_loss_fused(_p(image_all), _p(text_all), n, E, _p(idx_all), _p(temp), local_off, local_n, _p(work),
                               _p(loss), _p(di), _p(dt), _p(dtemp), stream_ptr()), "xfm_itc_loss_fused")
    return loss, di, dt, dtemp


def hard_negatives(image_feat, text_feat, temp, seed, idx=None, want_weights=False):
    B, E = image_feat.shape
    dev = image_feat.device
    w1 = torch.empty((B, B), dtype=torch.float32, device=dev) if want_weights else None
    w2 = torch.empty((B, B), dtype=torch.float32, device=dev) if want_weights else None
    tneg = torch.empty(B, dtype=torch.int64, device=dev)
    ineg = torch.empty(B, dtype=torch.int64, device=dev)
    check(lib().xfm_hard_negatives(_p(image_feat), _p(text_feat), B, E, _p(temp), _p(idx), C.c_uint64(seed), _p(w1),
                                   _p(w2), _p(tneg), _p(ineg), stream_ptr()), "xfm_hard_negatives")
    return ineg, tneg, w1, w2


def vq_argmin(z, codebook):
    R, Cd = z.shape
    assert z.dtype == torch.float32 and z.is_contiguous() and codebook.is_contiguous()
    ids = torch.empty(R, dtype=torch.int64, device=z.device)
    check(lib().xfm_vq_argmin(_p(z), _p(codebook), _p(ids), R, codebook.shape[0], Cd, stream_ptr()), "xfm_vq_argmin")
    return ids


def gelu_fwd(x):
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    check(lib().xfm_gelu_fwd(_p(x), _dt(x), _p(y), C.c_size_t(x.numel()), stream_ptr()), "xfm_gelu_fwd")
    return y


def gelu_bwd(dy, x):
    dx = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    check(lib().xfm_gelu_bwd(_p(dy), _dt(dy), _p(x), _dt(x), _p(dx), C.c_size_t(x.numel()), stream_ptr()), "xfm_gelu_bwd")
    return dx


def dropout_apply(x, p, seed):
    assert x.is_contiguous()
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    check(lib().xfm_dropout_apply(_p(x), _dt(x), _p(y), C.c_size_t(x.numel()), C.c_float(p), C.c_uint64(seed),
                                  stream_ptr()), "xfm_dropout_apply")
    return y


def l2norm_fwd(x):
    R, E = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous()
    y = torch.empty_like(x)
    inv = torch.empty(R, dtype=torch.float32, device=x.device)
    check(lib().xfm_l2norm_fwd(_p(x), _p(y), _p(inv), R, E, stream_ptr()), "xfm_l2norm_fwd")
    return y, inv


def l2norm_bwd(dy, y, inv):
    R, E = y.shape
    assert dy.dtype == torch.float32 and dy.is_contiguous()
    dx = torch.empty_like(y)
    check(lib().xfm_l2norm_bwd(_p(dy), _p(y), _p(inv), _p(dx), R, E, stream_ptr()), "xfm_l2norm_bwd")
    return dx


def mim_mse(x, t, mask_u8, with_cls=True):
    """x, t: f32 [B, np+1, D]; mask u8 [B, np].  Returns (loss[1], dx) for an upstream gradient of 1."""
    B, N, D = x.shape
    assert x.dtype == torch.float32 and t.dtype == torch.float32 and x.is_contiguous() and t.is_contiguous()
    assert mask_u8.dtype == torch.uint8 and mask_u8.is_contiguous() and mask_u8.shape == (B, N - 1)
    loss = torch.empty(1, dtype=torch.float32, device=x.device)
    count = torch.empty(1, dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x)
    check(lib().xfm_mim_mse(_p(x), _p(t), _p(mask_u8), B, N - 1, D, int(with_cls), _p(count), _p(loss), _p(dx),
                            stream_ptr()), "xfm_mim_mse")
    return loss, dx


def region_pool_fwd(y, idx, atts):
    """y f32 [n_img, N, D]; idx int64 [bsz]; atts int64 [bsz, N] -> (out f32 [bsz, N, D], out bf16)."""
    n_img, N, D = y.shape
    bsz = idx.numel()
    assert y.dtype == torch.float32 and y.is_contiguous() and idx.dtype == torch.int64 and atts.dtype == torch.int64
    assert atts.shape == (bsz, N) and atts.is_contiguous()
    out = torch.empty((bsz, N, D), dtype=torch.float32, device=y.device)
    out16 = torch.empty((bsz, N, D), dtype=torch.bfloat16, device=y.device)
    check(lib().xfm_region_pool_fwd(_p(y), _p(idx), _p(atts), _p(out), _p(out16), bsz, N, D, stream_ptr()), "xfm_region_pool_fwd")
    return out, out16


def region_pool_bwd_(dout, idx, atts, dy):
    bsz, N, D = dout.shape
    assert dout.dtype == torch.float32 and dout.is_contiguous() and dy.dtype == torch.float32 and dy.is_contiguous()
    check(lib().xfm_region_pool_bwd(_p(dout), _p(idx), _p(atts), _p(dy), bsz, N, D, stream_ptr()), "xfm_region_pool_bwd")


def sigmoid_fwd(x):
    assert x.dtype == torch.float32 and x.is_contiguous()
    y = torch.empty_like(x)
    check(lib().xfm_sigmoid_fwd(_p(x), _p(y), x.numel(), stream_ptr()), "xfm_sigmoid_fwd")
    return y


def sigmoid_bwd(dy, y):
    assert dy.dtype == torch.float32 and dy.is_contiguous() and y.is_contiguous()
    dx = torch.empty_like(y)
    check(lib().xfm_sigmoid_bwd(_p(dy), _p(y), _p(dx), y.numel(), stream_ptr()), "xfm_sigmoid_bwd")
    return dx


def bbox_loss(coord, target, is_image=None):
    """coord, target f32 [n, 4]; is_image f32 [n] or None.  Returns (loss_bbox[1], loss_giou[1], d_bbox [n,4], d_giou [n,4])."""
    n = coord.shape[0]
    assert coord.dtype == torch.float32 and coord.shape == (n, 4) and coord.is_contiguous()
    assert target.dtype == torch.float32 and target.shape == (n, 4) and target.is_contiguous()
    assert is_image is None or (is_image.dtype == torch.float32 and is_image.numel() == n and is_image.is_contiguous())
    dev = coord.device
    lb, lg = torch.empty(1, dtype=torch.float32, device=dev), torch.empty(1, dtype=torch.float32, device=dev)
    db, dg = torch.empty_like(coord), torch.empty_like(coord)
    check(lib().xfm_bbox_loss(_p(coord), _p(target), _p(is_image), n, _p(lb), _p(lg), _p(db), _p(dg), stream_ptr()),
          "xfm_bbox_loss")
    return lb, lg, db, dg


def image_u8_to_f32(img_u8, mean, std, flip=None, out=None):
    """ToTensor + Normalize (+ hflip) of dataset/__init__.py:26-35 on the device: img_u8 u8 [B, H, W, 3] -> f32 [B, 3, H, W]
    = (u8 / 255 - mean[c]) / std[c]; flip u8 [B] or None.  Bit-identical to the CPU transform."""
    assert img_u8.dtype == torch.uint8 and img_u8.dim() == 4 and img_u8.shape[3] == 3 and img_u8.is_contiguous()
    B, H, W, _ = img_u8.shape
    assert flip is None or (flip.dtype == torch.uint8 and flip.numel() == B and flip.is_contiguous())
    if out is None:
        out = torch.empty((B, 3, H, W), dtype=torch.float32, device=img_u8.device)
    assert out.dtype == torch.float32 and out.shape == (B, 3, H, W) and out.is_contiguous()
    m, s = (C.c_float * 3)(*[float(v) for v in mean]), (C.c_float * 3)(*[float(v) for v in std])
    check(lib().xfm_image_u8_to_f32(_p(img_u8), _p(out), _p(flip), B, H, W, m, s, stream_ptr()), "xfm_image_u8_to_f32")
    return out


def host_pack(tensors, out, threads=8):
    """Copy the bytes of the (contiguous, host) tensors or `bytes` objects back to back into `out` (uint8, host; normally pinned) with several
    threads.  Host-only: works without a CUDA device."""
    n = len(tensors)
    assert out.device.type == "cpu" and out.dtype == torch.uint8 and out.is_contiguous()
    assert all(isinstance(t, bytes) or (t.device.type == "cpu" and t.is_contiguous()) for t in tensors)
    srcs, nb = _host_segments(tensors)
    assert sum(nb) <= out.numel()
    check(load().xfm_host_pack(srcs, nb, n, C.c_void_p(out.data_ptr()), int(threads)), "xfm_host_pack")
    return out


def _host_segments(parts):
    """ctypes (void* [n], int64 [n]) of host tensors or `bytes` objects (their buffers, not copies; the caller keeps `parts`
    alive for the duration of the C call)."""
    n = len(parts)
    ptrs = [C.cast(C.c_char_p(p), C.c_void_p).value if isinstance(p, bytes) else p.data_ptr() for p in parts]
    sizes = [len(p) if isinstance(p, bytes) else p.numel() * p.element_size() for p in parts]
    return (C.c_void_p * max(n, 1))(*ptrs), (C.c_int64 * max(n, 1))(*sizes)


JPEG_INFO = 8      # XFM_JPEG_INFO: columns of xfm_jpeg_plan's per-image row


def jpeg_plan(blobs, threads=8):
    """Host-only marker walk of each `bytes` blob (xfm_jpeg_plan): int64 [n, 8] {status (0 = device path), width, height,
    restart intervals, coefficient blocks, plane bytes, 0, 0}.  Works without a CUDA device."""
    import numpy as np
    info = np.zeros((len(blobs), JPEG_INFO), np.int64)
    srcs, nb = _host_segments(blobs)
    check(load().xfm_jpeg_plan(srcs, nb, len(blobs), C.c_void_p(info.ctypes.data), int(threads)), "xfm_jpeg_plan")
    return info


def jpeg_tables(blobs, info, offs, threads=8):
    """Second host call (xfm_jpeg_tables): offs int64 [n, 4] {blob offset in the device byte buffer, first coefficient block,
    first plane byte, output byte offset}.  Returns (desc u8 [n * desc bytes], intervals int64 [sum info[:, 3], 2]) as host
    tensors, pinned when CUDA is there."""
    import numpy as np
    l = load()
    l.xfm_jpeg_desc_bytes.restype = C.c_size_t
    n = len(blobs)
    info, offs = np.ascontiguousarray(info, np.int64), np.ascontiguousarray(offs, np.int64)
    assert info.shape == (n, JPEG_INFO) and offs.shape == (n, 4)
    pin = torch.cuda.is_available()
    desc = torch.empty(max(n, 1) * l.xfm_jpeg_desc_bytes(), dtype=torch.uint8, pin_memory=pin)
    n_int = int(info[info[:, 0] == 0, 3].sum())
    intervals = torch.empty((max(n_int, 1), 2), dtype=torch.int64, pin_memory=pin)
    srcs, nb = _host_segments(blobs)
    check(l.xfm_jpeg_tables(srcs, nb, n, C.c_void_p(info.ctypes.data), C.c_void_p(offs.ctypes.data), C.c_void_p(desc.data_ptr()),
                            C.c_void_p(intervals.data_ptr()), int(threads)), "xfm_jpeg_tables")
    return desc, intervals


def jpeg_decode(data, desc, intervals, n, coef, planes, out, status, max_blocks, max_w, max_h):
    """The three decode launches (xfm_jpeg_decode) on the current stream; every tensor on the device (include/xfm_b200.h)."""
    assert data.dtype == torch.uint8 and desc.dtype == torch.uint8 and intervals.dtype == torch.int64 and coef.dtype == torch.int16
    assert planes.dtype == torch.uint8 and out.dtype == torch.uint8 and status.dtype == torch.int32 and status.numel() >= n
    check(lib().xfm_jpeg_decode(_p(data), _p(desc), _p(intervals), int(n), _p(coef), _p(planes), _p(out), _p(status),
                                C.c_int64(int(max_blocks)), int(max_w), int(max_h), stream_ptr()), "xfm_jpeg_decode")
    return out


def resize_taps(desc, out_h, out_w, KH, KV):
    """Pillow's bicubic tap tables for every image of desc (int64 [B, 8] device), computed on the device.
    Returns (hb, hk, vb, vk) for resize_bicubic_u8."""
    B = desc.shape[0]
    assert desc.dtype == torch.int64 and desc.shape == (B, 8) and desc.is_contiguous() and desc.is_cuda
    i32 = dict(dtype=torch.int32, device=desc.device)
    hb, hk = torch.empty((B, out_w, 2), **i32), torch.empty((B, out_w, KH), **i32)
    vb, vk = torch.empty((B, out_h, 2), **i32), torch.empty((B, out_h, KV), **i32)
    check(lib().xfm_resize_taps(_p(desc), _p(hb), _p(hk), KH, _p(vb), _p(vk), KV, B, out_h, out_w, stream_ptr()), "xfm_resize_taps")
    return hb, hk, vb, vk


def resize_bicubic_u8(src, desc, hb, hk, vb, vk, tmp, out, max_rows):
    """Crop + bicubic resize of ragged uint8 images (Pillow's ImagingResample; see include/xfm_b200.h).  src u8 packed; desc
    int64 [B, 8]; hb / vb int32 [B, OW|OH, 2]; hk / vk int32 [B, OW|OH, K]; tmp u8 scratch; out u8 [B, OH, OW, 3]."""
    B, OH, OW, _ = out.shape
    assert out.dtype == torch.uint8 and out.shape[3] == 3 and out.is_contiguous() and src.dtype == torch.uint8 and tmp.dtype == torch.uint8
    assert desc.dtype == torch.int64 and desc.shape == (B, 8) and desc.is_contiguous()
    for b_, k_, n_ in ((hb, hk, OW), (vb, vk, OH)):
        assert b_.dtype == torch.int32 and k_.dtype == torch.int32 and b_.shape == (B, n_, 2) and k_.shape[:2] == (B, n_)
        assert b_.is_contiguous() and k_.is_contiguous()
    check(lib().xfm_resize_bicubic_u8(_p(src), _p(desc), _p(hb), _p(hk), hk.shape[2], _p(vb), _p(vk), vk.shape[2], _p(tmp),
                                      _p(out), B, int(max_rows), OH, OW, stream_ptr()), "xfm_resize_bicubic_u8")
    return out


def axpby_scalars(a, sa, b, sb):
    """a * sa[0] + b * sb[0] (sa / sb: f32 [1] device tensors or None = 0)."""
    assert a.dtype == torch.float32 and a.is_contiguous() and b.is_contiguous() and a.shape == b.shape
    out = torch.empty_like(a)
    check(lib().xfm_axpby_scalars(_p(a), _p(sa), _p(b), _p(sb), _p(out), a.numel(), stream_ptr()), "xfm_axpby_scalars")
    return out


def adamw_hparams(lrs, wds, beta1, beta2, eps, max_grad_norm, grad_mul, correct_bias):
    """The 16-float hyper-parameter block of xfm_adamw_flat / xfm_grad_sumsq as a host tensor (pinned when CUDA is there)."""
    t = torch.tensor(list(lrs) + list(wds) + [beta1, beta2, eps, max_grad_norm, grad_mul, 1.0 if correct_bias else 0.0, 0.0, 0.0],
                     dtype=torch.float32)
    return t.pin_memory() if torch.cuda.is_available() else t


def grad_sumsq(G, chunk_seg, seg_group, seg_step, seg_bc, hp, out, accumulate=False):
    n = G.numel() // 64
    assert G.numel() % 64 == 0 and chunk_seg.numel() == n and chunk_seg.dtype == torch.int32
    assert seg_group.dtype == torch.uint8 and seg_step.dtype == torch.int32 and seg_bc.dtype == torch.float32
    assert seg_step.numel() == seg_group.numel() and seg_bc.numel() == 2 * seg_group.numel() and hp.numel() == 16
    check(lib().xfm_grad_sumsq(_p(G), _p(chunk_seg), _p(seg_group), C.c_size_t(n), _p(seg_step), _p(seg_bc),
                               seg_group.numel(), _p(hp), _p(out), int(accumulate), stream_ptr()), "xfm_grad_sumsq")


def adamw_flat(P, G, M, V, S, chunk_seg, seg_group, seg_bc, hp, sumsq=None, norm_out=None):
    n = P.numel() // 64
    assert P.numel() % 64 == 0 and chunk_seg.numel() == n and chunk_seg.dtype == torch.int32 and seg_group.dtype == torch.uint8
    check(lib().xfm_adamw_flat(_p(P), _p(G), _p(M), _p(V), _p(S), _p(chunk_seg), _p(seg_group), _p(seg_bc), C.c_size_t(n),
                               _p(sumsq), _p(norm_out), _p(hp), stream_ptr()), "xfm_adamw_flat")


def sgemm_f32(a, b, out=None, bias=None, accumulate=False):
    """Exact fp32 C[M,N] (+)= A[M,K] . B[N,K]^T (+ bias); a / b may be arbitrary-stride 2-D views (pass .t() for a transpose)."""
    assert a.dtype == torch.float32 and b.dtype == torch.float32 and a.dim() == 2 and b.dim() == 2
    M, K = a.shape
    N, Kb = b.shape
    assert K == Kb
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    assert out.shape == (M, N) and out.stride(1) == 1 and out.dtype == torch.float32
    check(lib().xfm_sgemm_f32(_p(a), C.c_int64(a.stride(0)), C.c_int64(a.stride(1)), _p(b), C.c_int64(b.stride(0)),
                              C.c_int64(b.stride(1)), _p(out), C.c_int64(out.stride(0)), M, N, K, _p(bias), int(accumulate),
                              stream_ptr()), "xfm_sgemm_f32")
    return out
