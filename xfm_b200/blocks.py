"""Forward / backward schedules of the encoder blocks, written against the C-ABI kernels (xfm_b200.lib).

No autograd inside: each *_fwd returns the tensors its *_bwd needs, and every parameter gradient is accumulated
straight into the flat gradient buffer (params.FlatParams.G).  The arithmetic follows
  * models/beit2.py:126-206   (pre-LN ViT block with LayerScale, relative position bias, DropPath),
  * models/vqkd_vit.py:122-199 (same block without LayerScale / bias, for the frozen VQ-KD tokenizer),
  * models/xroberta.py:201-304,358-473 (post-LN self-attn -> [cross-attn] -> FFN layer).
Residual streams that feed a LayerNorm stay fp32; GEMM operands are bf16; accumulation is fp32.
"""
import math

import torch

from . import lib as L


class Saved:
    """Bag of tensors kept for the backward pass."""
    pass


def _split_k(tiles, cap, kb):
    """Split-K factor for `tiles` output tiles on `cap` concurrent tile slots: the factor (<= 2 waves, >= 8 k-blocks per item)
    that fills whole waves best; ties go to the smaller factor (fewer fp32 atomics).  Measured on the step's shapes
    (tools/dev_wgrad.py): one full wave beats two half-length ones, e.g. 768 x 768 x 18912: 27.8 -> 23.8 us."""
    best, best_u = 1, 0.0
    for sk in range(1, max(1, min(2 * cap // max(tiles, 1), kb // 8)) + 1):
        items = tiles * sk
        u = items / (-(-items // cap) * cap)
        if u > best_u + 0.02:
            best, best_u = sk, u
    return best


def wgrad(fp_grad, dy, x):
    """fp_grad[Nout, Kin] += dy[T, Nout]^T · x[T, Kin]  (fp32 accumulate; split-K when few output tiles)."""
    T = dy.shape[0]
    n_out, k_in = fp_grad.shape
    kb = (T + 63) // 64
    if n_out >= L.PAIR_MIN_M and k_in >= 256:   # CTA-pair kernel: 256 x 256 tiles over 74 SM pairs
        split = _split_k(((n_out + 255) // 256) * ((k_in + 255) // 256), 74, kb)
        L.gemm(dy, x, a_t=True, b_t=True, out=fp_grad, accumulate=True, split_k=split)
    else:                                       # single-CTA kernel: 128 x 256 tiles over 148 SMs
        bn = 256 if k_in >= 256 else 0
        tiles = ((n_out + 127) // 128) * ((k_in + 255) // 256)
        L.gemm(dy, x, a_t=True, b_t=True, out=fp_grad, accumulate=True, split_k=_split_k(tiles, 148, kb), block_n=bn)


# =====================================================================================================
# BEiT / ViT block
# =====================================================================================================
def vit_block_fwd(x, w, B, N, H, eps, relbias=None, drop_scale=None, save=True, rel=None):
    """x: fp32 [B*N, D] residual stream.  w: dict of views for this block (see vision.py).  Returns (x_out, saved)."""
    D = x.shape[1]
    s = Saved() if save else None
    xn1, st1, _ = L.layernorm_fwd(x, w["n1w"], w["n1b"], eps, want_stats=save)
    qkv = L.gemm(xn1, w["qkv_w16"], bias=w["qkv_b"])
    attn, lse = L.attention_fwd(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], B, H, N, N, 0.125, bias=relbias,
                                rel_table=None if rel is None else rel[0], rel_window=0 if rel is None else rel[1])
    gamma1, gamma2 = w.get("g1"), w.get("g2")
    ds1, ds2 = drop_scale if isinstance(drop_scale, tuple) else (drop_scale, drop_scale)  # one DropPath draw per branch
    z1 = torch.empty_like(attn) if (save and gamma1 is not None) else None
    x1 = L.gemm(attn, w["proj_w16"], bias=w["proj_b"], col_scale=gamma1, row_group_scale=ds1, rows_per_group=N,
                residual=x, aux_out=z1, out_dtype=torch.float32)
    xn2, st2, _ = L.layernorm_fwd(x1, w["n2w"], w["n2b"], eps, want_stats=save)
    Fh = w["fc1_w16"].shape[0]
    h1 = torch.empty((x.shape[0], Fh), dtype=torch.bfloat16, device=x.device) if save else None
    a1 = L.gemm(xn2, w["fc1_w16"], bias=w["fc1_b"], act=1, aux_out=h1)
    z2 = torch.empty_like(attn) if (save and gamma2 is not None) else None
    x2 = L.gemm(a1, w["fc2_w16"], bias=w["fc2_b"], col_scale=gamma2, row_group_scale=ds2, rows_per_group=N,
                residual=x1, aux_out=z2, out_dtype=torch.float32)
    if save:
        s.x, s.st1, s.xn1, s.qkv, s.attn, s.lse, s.z1 = x, st1, xn1, qkv, attn, lse, z1
        s.x1, s.st2, s.xn2, s.h1, s.a1, s.z2 = x1, st2, xn2, h1, a1, z2
        s.relbias, s.ds1, s.ds2, s.rel = relbias, ds1, ds2, rel
    return x2, s


def vit_block_bwd(dx2, s, w, g, B, N, H, rel_index=None):
    """dx2: fp32 [B*N, D] gradient of the block output.  g: callable name -> fp32 grad view.  Returns dx (fp32)."""
    D = dx2.shape[1]
    dz2 = L.layerscale_bwd(dx2, s.z2, w["g2"], g("g2"), g("fc2_b"), s.ds2, N)
    wgrad(g("fc2_w"), dz2, s.a1)
    dh1 = L.gemm(dz2, w["fc2_w16"], b_t=True, act=2, aux_in=s.h1)
    L.colsum_into(dh1, g("fc1_b"))
    wgrad(g("fc1_w"), dh1, s.xn2)
    dxn2 = L.gemm(dh1, w["fc1_w16"], b_t=True)
    dx1 = L.layernorm_bwd(dxn2, s.x1, s.st2, w["n2w"], g("n2w"), g("n2b"), add_in=dx2)
    dz1 = L.layerscale_bwd(dx1, s.z1, w["g1"], g("g1"), g("proj_b"), s.ds1, N)
    wgrad(g("proj_w"), dz1, s.attn)
    dattn = L.gemm(dz1, w["proj_w16"], b_t=True)
    dqkv = torch.empty_like(s.qkv)
    ds = None
    tc = s.rel is not None and L.vit_attention_bwd_tc_ok(N)  # tcgen05 backward kernels (closed-form bias)
    if s.relbias is not None:
        ds = torch.empty((B, H, N, s.relbias.shape[2]), dtype=torch.bfloat16, device=dx2.device)
        if s.relbias.shape[2] != N and not tc:   # the tcgen05 kernel's TMA store writes the padding columns (zeros) itself
            ds[..., N:].zero_()
    q, k, v = s.qkv[:, :D], s.qkv[:, D:2 * D], s.qkv[:, 2 * D:]
    L.attention_bwd(dattn, q, k, v, s.attn, s.lse, B, H, N, N, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:],
                    bias=s.relbias, ds_dump=ds, rel_table=s.rel[0] if tc else None, rel_window=s.rel[1] if tc else 0)
    if ds is not None:
        dbias = L.batch_sum_bf16(ds)
        L.relpos_bias_bwd(dbias, rel_index, g("rel_table"), N, H, s.relbias.shape[2])
    L.colsum_into(dqkv[:, :D], g("q_bias"))
    L.colsum_into(dqkv[:, 2 * D:], g("v_bias"))
    wgrad(g("qkv_w"), dqkv, s.xn1)
    dxn1 = L.gemm(dqkv, w["qkv_w16"], b_t=True)
    return L.layernorm_bwd(dxn1, s.x, s.st1, w["n1w"], g("n1w"), g("n1b"), add_in=dx1)


# =====================================================================================================
# RoBERTa layer (self-attn -> [cross-attn] -> FFN), post-LN
# =====================================================================================================
class DropCfg:
    """Dropout state of one forward pass: probabilities and a counter-derived seed per site."""

    def __init__(self, p_hidden=0.0, p_attn=0.0, seed=0):
        self.p_hidden, self.p_attn, self.seed, self._n = p_hidden, p_attn, seed, 0

    def next_seed(self):
        self._n += 1
        return (self.seed * 1000003 + self._n * 7919) & 0x7FFFFFFFFFFFFFFF


NO_DROP = DropCfg()


def _attn_out_fwd(ctx, w, pre, resid, eps, drop, s, tag):
    """RobertaSelfOutput (xroberta.py:300-304): LayerNorm(dropout(dense(ctx)) + resid).  Returns (bf16, f32) copies of the
    LayerNorm output: the bf16 one feeds the next GEMM, the f32 one is the next residual."""
    seed = drop.next_seed() if drop.p_hidden > 0 else 0
    pre_ln = L.gemm(ctx, w[pre + "o_w16"], bias=w[pre + "o_b"], dropout_p=drop.p_hidden, dropout_seed=seed, residual=resid,
                    out_dtype=torch.float32)
    h, st, h32 = L.layernorm_fwd(pre_ln, w[pre + "ln_w"], w[pre + "ln_b"], eps, want_f32_copy=True, want_stats=s is not None)
    if s is not None:
        setattr(s, tag + "_pre_ln", pre_ln)
        setattr(s, tag + "_st", st)
        setattr(s, tag + "_seed", seed)
    return h, h32


def roberta_layer_fwd(h, w, Bt, Lt, H, eps, kmask, enc=None, Benc=0, Lenc=0, kv_index=None, drop=NO_DROP, save=True,
                      h32=None, kv_offsets=None, kv_samples=None, self_bias=None, enc_kmask=None, kvc=None, varlen=None):
    """h: bf16 [Bt*Lt, D] (h32: the same hidden state in f32, used as the residual when given).
    varlen: encoders.Varlen of a packed variable-length batch (h holds its T rows; Bt, Lt and kmask are unused): the
    self-attention runs on the packed kernels, everything else is row-wise anyway.
    enc: bf16 [Benc*Lenc, Denc] image tokens (cross-attention) or None.  Returns (h_out bf16, h_out f32, saved).
    self_bias: f32 [H, Lt, ld] additive self-attention term (the decoder's causal mask, xroberta.py:771-806);
    enc_kmask: f32 [Bt, Lenc] additive key mask of the cross-attention (xroberta.py:903-909).
    kvc: this layer's cross-attention K | V projection of `enc` when the caller computed it for all layers in one GEMM (a
    column slice of that GEMM's output, encoders.RobertaStack.layers_fwd)."""
    D = h.shape[1]
    s = Saved() if save else None
    scale = 1.0 / math.sqrt(64)
    qkv = L.gemm(h, w["qkv_w16"], bias=w["qkv_b"])
    seed_a = drop.next_seed() if drop.p_attn > 0 else 0
    if varlen is not None:
        ctx, lse = L.attention_varlen_fwd(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], varlen.cu, varlen.tiles, H, varlen.Lpad,
                                          scale, dropout_p=drop.p_attn, dropout_seed=seed_a)
    else:
        ctx, lse = L.attention_fwd(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], Bt, H, Lt, Lt, scale, kmask=kmask,
                                   bias=self_bias, dropout_p=drop.p_attn, dropout_seed=seed_a)
    h1, h1_32 = _attn_out_fwd(ctx, w, "a_", h if h32 is None else h32, eps, drop, s, "a")
    if save:
        s.h, s.qkv, s.ctx, s.lse, s.seed_a, s.h1 = h, qkv, ctx, lse, seed_a, h1
        s.p_hidden, s.p_attn = drop.p_hidden, drop.p_attn
    h2, h2_32 = h1, h1_32
    if enc is not None:
        qc = L.gemm(h1, w["c_q_w16"], bias=w["c_q_b"])
        if kvc is None:
            kvc = L.gemm(enc, w["c_kv_w16"], bias=w["c_kv_b"])
        seed_c = drop.next_seed() if drop.p_attn > 0 else 0
        cctx, clse = L.attention_fwd(qc, kvc[:, :D], kvc[:, D:], Bt, H, Lt, Lenc, scale, Bkv=Benc, kv_index=kv_index,
                                     kmask=enc_kmask, dropout_p=drop.p_attn, dropout_seed=seed_c, kv_offsets=kv_offsets,
                                     kv_samples=kv_samples)
        h2, h2_32 = _attn_out_fwd(cctx, w, "c_", h1_32, eps, drop, s, "c")
        if save:
            s.qc, s.kvc, s.cctx, s.clse, s.seed_c, s.h2, s.enc = qc, kvc, cctx, clse, seed_c, h2, enc
    Fh = w["i_w16"].shape[0]
    pre = torch.empty((h.shape[0], Fh), dtype=torch.bfloat16, device=h.device) if save else None
    act = L.gemm(h2, w["i_w16"], bias=w["i_b"], act=1, aux_out=pre)
    seed_f = drop.next_seed() if drop.p_hidden > 0 else 0
    pre_ln = L.gemm(act, w["f_w16"], bias=w["f_b"], dropout_p=drop.p_hidden, dropout_seed=seed_f, residual=h2_32,
                    out_dtype=torch.float32)
    h3, st3, h3_32 = L.layernorm_fwd(pre_ln, w["f_ln_w"], w["f_ln_b"], eps, want_f32_copy=True, want_stats=save)
    if save:
        s.pre, s.act, s.f_pre_ln, s.f_st, s.f_seed, s.has_cross = pre, act, pre_ln, st3, seed_f, enc is not None
    return h3, h3_32, s


def _bf16_copy(x32):
    x16 = torch.empty(x32.shape, dtype=torch.bfloat16, device=x32.device)
    L.cast_to_bf16(x32, x16)
    return x16


def _attn_out_bwd(dh, s, w, g, pre, tag, ctx):
    """Backward of LayerNorm(dropout(dense(ctx)) + resid).  Returns (d_pre_ln f32 = grad wrt resid, d_ctx bf16).
    The residual-stream gradient stays fp32 between layers: LayerNorm backward cancels the large mean / x-hat components
    of dy, so bf16 rounding of dy would dominate the small components that survive."""
    d_pre, d_dense = L.layernorm_bwd_dense(dh, getattr(s, tag + "_pre_ln"), getattr(s, tag + "_st"), w[pre + "ln_w"],
                                           g(pre + "ln_w"), g(pre + "ln_b"), g(pre + "o_b"), drop_p=s.p_hidden,
                                           drop_seed=getattr(s, tag + "_seed"))
    wgrad(g(pre + "o_w"), d_dense, ctx)
    d_ctx = L.gemm(d_dense, w[pre + "o_w16"], b_t=True)
    return d_pre, d_ctx


def roberta_layer_bwd(dh3, s, w, g, Bt, Lt, H, kmask, Benc=0, Lenc=0, kv_index=None, kv_offsets=None, kv_samples=None,
                      d_enc=None, need_dh=True, self_bias=None, enc_kmask=None, dkvc_out=None, varlen=None):
    """dh3: bf16 or fp32 [Bt*Lt, D].  d_enc: fp32 [Benc*Lenc, Denc] accumulator for the image-token gradient.
    dkvc_out: where this layer's K | V gradient goes when the caller back-propagates all layers' K / V projections in one
    GEMM afterwards (the per-layer d_enc GEMM is then skipped).  Returns the fp32 gradient wrt the layer input (or None)."""
    D = s.h.shape[1]
    scale = 1.0 / math.sqrt(64)
    f32 = torch.float32
    # ---- FFN
    d_pre_ln, d_dense = L.layernorm_bwd_dense(dh3, s.f_pre_ln, s.f_st, w["f_ln_w"], g("f_ln_w"), g("f_ln_b"), g("f_b"),
                                              drop_p=s.p_hidden, drop_seed=s.f_seed)
    wgrad(g("f_w"), d_dense, s.act)
    d_i = L.gemm(d_dense, w["f_w16"], b_t=True, act=2, aux_in=s.pre)
    L.colsum_into(d_i, g("i_b"))
    h2 = s.h2 if s.has_cross else s.h1
    wgrad(g("i_w"), d_i, h2)
    dh2 = L.gemm(d_i, w["i_w16"], b_t=True, residual=d_pre_ln, out_dtype=f32)
    # ---- cross-attention
    dh1 = dh2
    if s.has_cross:
        d_res, d_cctx = _attn_out_bwd(dh2, s, w, g, "c_", "c", s.cctx)
        dqc = torch.empty_like(s.qc)
        dkvc = torch.empty_like(s.kvc) if dkvc_out is None else dkvc_out
        L.attention_bwd(d_cctx, s.qc, s.kvc[:, :D], s.kvc[:, D:], s.cctx, s.clse, Bt, H, Lt, Lenc, scale, dqc, dkvc[:, :D],
                        dkvc[:, D:], Bkv=Benc, kv_index=kv_index, kv_offsets=kv_offsets, kv_samples=kv_samples,
                        kmask=enc_kmask, dropout_p=s.p_attn, dropout_seed=s.seed_c)
        L.colsum_into(dqc, g("c_q_b"))
        wgrad(g("c_q_w"), dqc, s.h1)
        dh1 = L.gemm(dqc, w["c_q_w16"], b_t=True, residual=d_res, out_dtype=f32)
        L.colsum_into(dkvc, g("c_kv_b"))
        wgrad(g("c_kv_w"), dkvc, s.enc)
        if d_enc is not None and dkvc_out is None:
            L.gemm(dkvc, w["c_kv_w16"], b_t=True, out=d_enc, accumulate=True)
    # ---- self-attention
    d_res, d_ctx = _attn_out_bwd(dh1, s, w, g, "a_", "a", s.ctx)
    dqkv = torch.empty_like(s.qkv)
    if varlen is not None:
        L.attention_varlen_bwd(d_ctx, s.qkv[:, :D], s.qkv[:, D:2 * D], s.qkv[:, 2 * D:], s.ctx, s.lse, varlen.cu, varlen.tiles, H,
                               varlen.Lpad, scale, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], dropout_p=s.p_attn,
                               dropout_seed=s.seed_a)
    else:
        L.attention_bwd(d_ctx, s.qkv[:, :D], s.qkv[:, D:2 * D], s.qkv[:, 2 * D:], s.ctx, s.lse, Bt, H, Lt, Lt, scale,
                        dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], kmask=kmask, bias=self_bias, dropout_p=s.p_attn,
                        dropout_seed=s.seed_a)
    L.colsum_into(dqkv, g("qkv_b"))
    wgrad(g("qkv_w"), dqkv, s.h)
    if not need_dh:
        return None
    return L.gemm(dqkv, w["qkv_w16"], b_t=True, residual=d_res, out_dtype=f32)
