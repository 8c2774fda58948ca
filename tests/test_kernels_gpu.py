"""Kernel-level parity: every C-ABI entry point against the CPU oracle / a plain fp32 PyTorch restatement of the
same op on the same seeded inputs.  Tolerances: bit-exact for integer outputs; bf16-rounding bounds for
floating-point kernels (stated per test)."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import xfm_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from xfm_b200 import lib as L

    L.lib()
    return L


def G(seed=0):
    return torch.Generator(device="cpu").manual_seed(seed)


def bf(x):
    return x.to(torch.bfloat16)


def rel_err(a, b):
    return float((a.float().cpu() - b.float().cpu()).abs().max() / b.float().abs().max().clamp_min(1e-6))


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K,a_t,b_t", [(788, 200, 72, False, False), (256, 768, 768, False, True),
                                           (768, 768, 4000, True, True), (96, 2, 1536, False, False),
                                           (1000, 2304, 768, False, False)])
def test_gemm_layouts(lib, M, N, K, a_t, b_t):
    g = G(M + N)
    A, B = bf(torch.randn(M, K, generator=g)), bf(torch.randn(N, K, generator=g))
    ref = A.float() @ B.float().t()
    a = (A.t().contiguous() if a_t else A).cuda()
    b = (B.t().contiguous() if b_t else B).cuda()
    out = lib.gemm(a, b, a_t=a_t, b_t=b_t, out_dtype=torch.float32)
    assert rel_err(out, ref) < 1e-5  # fp32 accumulate of exact bf16 products
    out16 = lib.gemm(a, b, a_t=a_t, b_t=b_t)
    assert rel_err(out16, ref) < 5e-3  # one bf16 rounding of the result


def test_gemm_epilogues(lib):
    g = G(3)
    M, N, K = 394, 768, 256
    A, B = bf(torch.randn(M, K, generator=g)), bf(torch.randn(N, K, generator=g) * 0.1)
    bias, gamma = torch.randn(N, generator=g), torch.randn(N, generator=g)
    rs = torch.rand(2, generator=g)
    res = torch.randn(M, N, generator=g)
    z = A.float() @ B.float().t() + bias
    ref = res + z * gamma * rs.repeat_interleave(197)[:, None]
    aux = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    out = lib.gemm(A.cuda(), B.cuda(), bias=bias.cuda(), col_scale=gamma.cuda(), row_group_scale=rs.cuda(),
                   rows_per_group=197, residual=res.cuda(), aux_out=aux, out_dtype=torch.float32)
    assert rel_err(out, ref) < 1e-5
    assert rel_err(aux, z) < 5e-3
    # GELU forward with pre-activation copy, then the dGELU epilogue
    out = lib.gemm(A.cuda(), B.cuda(), bias=bias.cuda(), act=1, aux_out=aux)
    assert rel_err(out, F.gelu(z)) < 5e-3
    h = bf(torch.randn(M, N, generator=g))
    hf = h.float()
    dgelu = 0.5 * (1 + torch.erf(hf / math.sqrt(2))) + hf * torch.exp(-0.5 * hf * hf) / math.sqrt(2 * math.pi)
    out = lib.gemm(A.cuda(), B.cuda(), act=2, aux_in=h.cuda(), out_dtype=torch.float32)
    assert rel_err(out, (A.float() @ B.float().t()) * dgelu) < 1e-4
    # split-K accumulate into an existing f32 buffer (wgrad)
    acc = torch.randn(N, K, generator=g)
    X = bf(torch.randn(M, N, generator=g))  # dY [tokens, N]
    ref = acc + X.float().t() @ A.float()
    out = acc.clone().cuda()
    lib.gemm(X.cuda(), A.cuda(), a_t=True, b_t=True, out=out, accumulate=True, split_k=4)
    assert rel_err(out, ref) < 1e-5


@pytest.mark.parametrize("M,N,K", [(2560, 768, 256), (2500, 304, 200), (2049, 1000, 64)])
def test_gemm_cta_pair_epilogues(lib, M, N, K):
    """CTA-pair (cta_group::2) kernel (selected for M >= 2048, N >= 256): every epilogue mode on
    full and ragged tiles (M, N not multiples of the 256 x 256 tile / the 32 x 32 epilogue block), against the single-CTA
    kernel (block_n = 128) and against fp32 torch."""
    g = G(M + N + K)
    A, B = bf(torch.randn(M, K, generator=g)), bf(torch.randn(N, K, generator=g) * 0.1)
    bias, gamma = torch.randn(N, generator=g), torch.randn(N, generator=g)
    rpg = 197
    rs = torch.rand((M + rpg - 1) // rpg, generator=g)
    res = torch.randn(M, N, generator=g)
    z = A.float() @ B.float().t() + bias
    ref = res + z * gamma * rs.repeat_interleave(rpg)[:M, None]
    Ad, Bd = A.cuda(), B.cuda()
    for bn in (0, 128):   # 0 = automatic: the pair kernel at these sizes
        aux = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
        out = lib.gemm(Ad, Bd, bias=bias.cuda(), col_scale=gamma.cuda(), row_group_scale=rs.cuda(), rows_per_group=rpg,
                       residual=res.cuda(), aux_out=aux, out_dtype=torch.float32, block_n=bn)
        assert rel_err(out, ref) < 1e-5, bn
        assert rel_err(aux, z) < 5e-3, bn
        out = lib.gemm(Ad, Bd, bias=bias.cuda(), act=1, aux_out=aux, block_n=bn)
        assert rel_err(out, F.gelu(z)) < 5e-3, bn
        assert rel_err(aux, z) < 5e-3, bn
        h = bf(torch.randn(M, N, generator=G(7)))
        hf = h.float()
        dgelu = 0.5 * (1 + torch.erf(hf / math.sqrt(2))) + hf * torch.exp(-0.5 * hf * hf) / math.sqrt(2 * math.pi)
        out = lib.gemm(Ad, Bd, act=2, aux_in=h.cuda(), block_n=bn)
        assert rel_err(out, (A.float() @ B.float().t()) * dgelu) < 5e-3, bn
        # dropout + f32 residual -> f32 (text layers); the two kernels must drop the same elements
        d = lib.gemm(Ad, Bd, bias=bias.cuda(), dropout_p=0.1, dropout_seed=3, residual=res.cuda(), out_dtype=torch.float32,
                     block_n=bn)
        kept = (d - res.cuda()) != 0
        assert abs(float(kept.float().mean()) - 0.9) < 0.01
        assert rel_err((d - res.cuda())[kept], (z.cuda() / 0.9)[kept]) < 1e-4
        if bn == 0:
            d_pair = d
        else:
            assert torch.equal(d_pair != res.cuda(), d != res.cuda())
    acc = torch.randn(N, K, generator=g)
    X = bf(torch.randn(M, N, generator=g))
    out = acc.clone().cuda()
    lib.gemm(X.cuda(), Ad, a_t=True, b_t=True, out=out, accumulate=True, split_k=3)
    assert rel_err(out, acc + X.float().t() @ A.float()) < 1e-5


@pytest.mark.parametrize("M,N,K", [(2560, 768, 256), (2500, 288, 200), (4000, 1536, 128), (18912, 768, 768)])
def test_gemm_cta_pair_f32_tma_epilogue(lib, M, N, K):
    """f32 TMA epilogue of the CTA-pair kernel (f32 residual in through TMA, f32 out through TMA, N % 32 == 0): LayerScale /
    DropPath scales, dropout, plain f32 output and the MN-major (dgrad) operand, on full and ragged M / N tiles, against
    fp32 torch and against the single-CTA kernel's generic epilogue (same dropout decisions)."""
    g = G(3 * M + N + K)
    A, B = bf(torch.randn(M, K, generator=g)), bf(torch.randn(N, K, generator=g) * 0.1)
    bias, gamma = torch.randn(N, generator=g), torch.randn(N, generator=g)
    rpg = 197
    rs = torch.rand((M + rpg - 1) // rpg, generator=g)
    res = torch.randn(M, N, generator=g)
    z = A.float() @ B.float().t()
    Ad, Bd, resd = A.cuda(), B.cuda(), res.cuda()
    out = lib.gemm(Ad, Bd, bias=bias.cuda(), col_scale=gamma.cuda(), row_group_scale=rs.cuda(), rows_per_group=rpg,
                   residual=resd, out_dtype=torch.float32)
    assert rel_err(out, res + (z + bias) * gamma * rs.repeat_interleave(rpg)[:M, None]) < 1e-5
    aux = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device="cuda")   # ViT blocks: saved pre-scale value
    out2 = lib.gemm(Ad, Bd, bias=bias.cuda(), col_scale=gamma.cuda(), row_group_scale=rs.cuda(), rows_per_group=rpg,
                    residual=resd, aux_out=aux, out_dtype=torch.float32)
    assert torch.equal(out, out2) and rel_err(aux, z + bias) < 5e-3
    out = lib.gemm(Ad, Bd, out_dtype=torch.float32)                      # no bias, no residual
    assert rel_err(out, z) < 1e-5
    out = lib.gemm(Ad, Bd, bias=bias.cuda(), residual=resd, out_dtype=torch.float32)
    assert rel_err(out, z + bias + res) < 1e-5
    d_pair = lib.gemm(Ad, Bd, bias=bias.cuda(), dropout_p=0.1, dropout_seed=11, residual=resd, out_dtype=torch.float32)
    d_one = lib.gemm(Ad, Bd, bias=bias.cuda(), dropout_p=0.1, dropout_seed=11, residual=resd, out_dtype=torch.float32,
                     block_n=128)
    kept = (d_pair - resd) != 0
    assert abs(float(kept.float().mean()) - 0.9) < 0.01
    assert torch.equal(kept, (d_one - resd) != 0)
    assert rel_err(d_pair, d_one) < 1e-6
    # dgrad form: B stored [K, N] (MN-major), f32 residual = gradient of the skip connection
    Bt = B.t().contiguous().cuda()
    out = lib.gemm(Ad, Bt, b_t=True, residual=resd, out_dtype=torch.float32)
    assert rel_err(out, z + res) < 1e-5
    # dGELU TMA epilogue (pre-activation tile in through TMA, bf16 result written in place and stored by TMA)
    h = bf(torch.randn(M, N, generator=G(7)))
    hf = h.float()
    dgelu = 0.5 * (1 + torch.erf(hf / math.sqrt(2))) + hf * torch.exp(-0.5 * hf * hf) / math.sqrt(2 * math.pi)
    out = lib.gemm(Ad, Bt, b_t=True, act=2, aux_in=h.cuda())
    assert rel_err(out, z * dgelu) < 5e-3
    assert torch.equal(out, lib.gemm(Ad, Bt, b_t=True, act=2, aux_in=h.cuda(), block_n=128))
    # output written into a strided view (row stride > N)
    wide = torch.zeros(M, N + 64, dtype=torch.float32, device="cuda")
    lib.gemm(Ad, Bd, bias=bias.cuda(), residual=resd, out=wide[:, :N])
    assert rel_err(wide[:, :N], z + bias + res) < 1e-5 and float(wide[:, N:].abs().max()) == 0.0


def test_gemm_dropout_statistics_and_determinism(lib):
    g = G(5)
    A, B = bf(torch.randn(512, 64, generator=g)), bf(torch.randn(256, 64, generator=g))
    a = lib.gemm(A.cuda(), B.cuda(), dropout_p=0.1, dropout_seed=77, out_dtype=torch.float32)
    b = lib.gemm(A.cuda(), B.cuda(), dropout_p=0.1, dropout_seed=77, out_dtype=torch.float32)
    assert torch.equal(a, b)
    ref = (A.float() @ B.float().t()).cuda()
    kept = a != 0
    assert abs(float(kept.float().mean()) - 0.9) < 0.01
    assert rel_err(a[kept], ref[kept] / 0.9) < 1e-5


# ------------------------------------------------------------------------------------------------ LayerNorm
@pytest.mark.parametrize("D,xd", [(768, torch.float32), (768, torch.bfloat16), (128, torch.float32), (1536, torch.float32),
                                  (3072, torch.float32)])   # 3072: build_mlp on two concatenated CLS rows (model_nlvr.py:25)
def test_layernorm_fwd_bwd(lib, D, xd):
    g = G(D)
    M = 333
    x = (torch.randn(M, D, generator=g) * 2 + 0.5).to(xd)
    w, b = 1 + 0.1 * torch.randn(D, generator=g), 0.1 * torch.randn(D, generator=g)
    dy = torch.randn(M, D, generator=g)
    add = torch.randn(M, D, generator=g)
    xr = x.float().requires_grad_(True)
    wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = F.layer_norm(xr, (D,), wr, br, 1e-5)
    ref.backward(dy)
    y, stats, y2 = lib.layernorm_fwd(x.cuda(), w.cuda(), b.cuda(), 1e-5, want_f32_copy=True)
    assert rel_err(y2, ref) < 2e-6
    assert rel_err(y, ref) < 5e-3
    dw, db = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    dx = lib.layernorm_bwd(dy.cuda(), x.cuda(), stats, w.cuda(), dw, db, add_in=add.cuda())
    assert rel_err(dx, xr.grad + add) < 1e-5
    assert rel_err(dw, wr.grad) < 1e-5 and rel_err(db, br.grad) < 1e-5


@pytest.mark.parametrize("M,p", [(333, 0.0), (3840, 0.1), (15360, 0.1)])
def test_layernorm_bwd_dense_equals_the_three_pass_form(lib, M, p):
    """xfm_layernorm_bwd_dense = layernorm_bwd, then dropout_apply (or the bf16 cast) of its output, then the bias column
    sum of that: dx bit-equal, the bf16 copy bit-equal (same mask as the GEMM epilogue's), column sums to fp32 rounding."""
    D = 768
    g = G(M)
    x = torch.randn(M, D, generator=g) * 2 + 0.5
    w, b = 1 + 0.1 * torch.randn(D, generator=g), 0.1 * torch.randn(D, generator=g)
    dy = torch.randn(M, D, generator=g)
    _, stats, _ = lib.layernorm_fwd(x.cuda(), w.cuda(), b.cuda(), 1e-5)
    dw0, db0 = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    dx0 = lib.layernorm_bwd(dy.cuda(), x.cuda(), stats, w.cuda(), dw0, db0)
    if p > 0:
        d16_0 = lib.dropout_apply(dx0, p, 77)
    else:
        d16_0 = dx0.to(torch.bfloat16)
    bias0 = torch.zeros(D, device="cuda")
    lib.colsum_into(d16_0, bias0)
    dw1, db1, bias1 = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    dx1, d16_1 = lib.layernorm_bwd_dense(dy.cuda(), x.cuda(), stats, w.cuda(), dw1, db1, bias1, drop_p=p, drop_seed=77)
    assert torch.equal(dx0, dx1) and torch.equal(d16_0, d16_1)
    assert rel_err(dw1, dw0) < 1e-5 and rel_err(db1, db0) < 1e-5 and rel_err(bias1, bias0) < 1e-5
    if p > 0:
        assert abs(float((d16_1 != 0).float().mean()) - (1 - p)) < 0.01


@pytest.mark.parametrize("dyd", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("with_add", [False, True])
@pytest.mark.parametrize("dense", [False, True])
def test_layernorm_bwd_specialised_instantiations(lib, dyd, with_add, dense):
    """D = 768 with fp32 x / dx runs the dtype-specialised instantiations of layernorm_bwd_kernel (elementwise.cu, DT >= 0):
    every one of them against torch autograd, ragged row count (the last CTA and the last warps have fewer rows)."""
    if dense and with_add:
        pytest.skip("the dense form has no add_in")
    D, M = 768, 1237
    g = G(31 + int(with_add) + 2 * int(dense))
    x = torch.randn(M, D, generator=g) * 2 + 0.5
    w, b = 1 + 0.1 * torch.randn(D, generator=g), 0.1 * torch.randn(D, generator=g)
    dy = torch.randn(M, D, generator=g).to(dyd)
    add = torch.randn(M, D, generator=g) if with_add else None
    xr = x.clone().requires_grad_(True)
    wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    F.layer_norm(xr, (D,), wr, br, 1e-5).backward(dy.float())
    want = xr.grad + (add if with_add else 0)
    _, stats, _ = lib.layernorm_fwd(x.cuda(), w.cuda(), b.cuda(), 1e-5)
    dw, db = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    if dense:
        dbias = torch.zeros(D, device="cuda")
        dx, dx16 = lib.layernorm_bwd_dense(dy.cuda(), x.cuda(), stats, w.cuda(), dw, db, dbias)
        assert torch.equal(dx16, dx.to(torch.bfloat16))
        assert rel_err(dbias, dx16.float().sum(0)) < 1e-5
    else:
        dx = lib.layernorm_bwd(dy.cuda(), x.cuda(), stats, w.cuda(), dw, db, add_in=None if add is None else add.cuda())
    assert rel_err(dx, want) < 1e-5
    assert rel_err(dw, wr.grad) < 1e-5 and rel_err(db, br.grad) < 1e-5


def test_layerscale_bwd_and_colsum(lib):
    g = G(9)
    M, D = 394, 768
    dxo, z = torch.randn(M, D, generator=g), bf(torch.randn(M, D, generator=g))
    gamma, rs = torch.randn(D, generator=g), torch.rand(2, generator=g)
    s = rs.repeat_interleave(197)[:, None]
    dgamma, dbias = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    dz = lib.layerscale_bwd(dxo.cuda(), z.cuda(), gamma.cuda(), dgamma, dbias, rs.cuda(), 197)
    ref_dz = dxo * gamma * s
    assert rel_err(dz, ref_dz) < 5e-3
    assert rel_err(dgamma, (dxo * s * z.float()).sum(0)) < 1e-5
    assert rel_err(dbias, ref_dz.sum(0)) < 1e-5
    big = bf(torch.randn(1000, 2304, generator=g))
    out = torch.zeros(768, device="cuda")
    lib.colsum_into(big.cuda()[:, 1536:], out)  # strided view, like the v-bias gradient
    assert rel_err(out, big.float()[:, 1536:].sum(0)) < 1e-5


# ------------------------------------------------------------------------------------------------ embeddings / patches
def test_roberta_embeddings(lib):
    cfg = O.tiny_config()
    sd = O.make_state_dict(cfg)
    batch = O.make_batch(cfg, 5, L=24, M=6)
    p = "text_encoder.roberta.embeddings."
    ref = O.roberta_embeddings(batch["text_ids"], sd, "text_encoder.", cfg)
    c = {k: v.cuda() for k, v in sd.items() if k.startswith(p)}
    y, pre, stats, pos_ids = lib.roberta_embed_fwd(batch["text_ids"].cuda(), c[p + "word_embeddings.weight"],
                                                   c[p + "position_embeddings.weight"], c[p + "token_type_embeddings.weight"],
                                                   c[p + "LayerNorm.weight"], c[p + "LayerNorm.bias"], cfg["pad_id"], cfg["ln_eps"])
    assert torch.equal(pos_ids.cpu().long(), O.roberta_position_ids(batch["text_ids"], cfg["pad_id"]))  # bit-exact ids
    assert rel_err(y.view(ref.shape), ref) < 5e-3
    # backward scatter
    g = G(1)
    dpre = torch.randn(5 * 24, cfg["hidden"], generator=g)
    word = sd[p + "word_embeddings.weight"].clone().requires_grad_(True)
    pos = sd[p + "position_embeddings.weight"].clone().requires_grad_(True)
    typ = sd[p + "token_type_embeddings.weight"].clone().requires_grad_(True)
    pid = O.roberta_position_ids(batch["text_ids"], cfg["pad_id"])
    e = F.embedding(batch["text_ids"], word, padding_idx=cfg["pad_id"]) + typ[0] + F.embedding(pid, pos, padding_idx=cfg["pad_id"])
    e.view(-1, cfg["hidden"]).backward(dpre)
    dword, dpos, dtyp = torch.zeros_like(word).cuda(), torch.zeros_like(pos).cuda(), torch.zeros(cfg["hidden"]).cuda()
    lib.roberta_embed_bwd(dpre.cuda(), batch["text_ids"].cuda(), pos_ids, dword, dpos, dtyp, cfg["pad_id"])
    assert rel_err(dword, word.grad) < 1e-5 and rel_err(dpos, pos.grad) < 1e-5 and rel_err(dtyp, typ.grad[0]) < 1e-5


def test_patch_pipeline(lib):
    g = G(2)
    B, P, res, D = 3, 16, 64, 128
    img = torch.randn(B, 3, res, res, generator=g)
    W, bias = torch.randn(D, 3, P, P, generator=g) * 0.05, torch.randn(D, generator=g)
    ref = F.conv2d(bf(img).float(), bf(W).float(), bias, stride=P).flatten(2).transpose(1, 2)
    cols = lib.im2col(img.cuda(), P)
    patch = lib.gemm(cols, bf(W.view(D, -1)).cuda(), bias=bias.cuda(), out_dtype=torch.float32)
    assert rel_err(patch.view(B, -1, D), ref) < 1e-5
    npatch = ref.shape[1]
    mask = torch.rand(B, npatch, generator=g) < 0.4
    cls, mtok = torch.randn(D, generator=g), torch.randn(D, generator=g)
    x = lib.assemble_tokens(patch, cls.cuda(), mtok.cuda(), mask.to(torch.uint8).cuda(), None, B, npatch)
    w = mask.unsqueeze(-1).float()
    want = torch.cat([cls.expand(B, 1, D), patch.cpu().view(B, npatch, D) * (1 - w) + mtok * w], 1)
    assert torch.equal(x.cpu().view(B, npatch + 1, D), want)
    dx = torch.randn(B * (npatch + 1), D, generator=g)
    dcls, dm = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    dpatch = lib.assemble_tokens_bwd(dx.cuda(), mask.to(torch.uint8).cuda(), dcls, dm, B, npatch)
    d3 = dx.view(B, npatch + 1, D)
    assert rel_err(dcls, d3[:, 0].sum(0)) < 1e-5
    assert rel_err(dm, (d3[:, 1:] * w).sum((0, 1))) < 1e-5
    assert rel_err(dpatch.view(B, npatch, D), d3[:, 1:] * (1 - w)) < 5e-3
    # VQ-KD pre-processing folded into im2col
    img01 = torch.rand(B, 3, res, res, generator=g)
    c2 = lib.im2col(img01.cuda(), P, pre_mul=torch.tensor([255.0], device="cuda"))
    ref2 = F.unfold(O.vqkd_preprocess(img01), P, stride=P).transpose(1, 2).reshape(-1, 3 * P * P)
    assert rel_err(c2, ref2) < 5e-3


def test_meanpool_gather_scatter_relpos(lib):
    g = G(4)
    B, npatch, D = 3, 16, 128
    y32 = torch.randn(B * (npatch + 1), D, generator=g).cuda()
    y16 = y32.to(torch.bfloat16)
    ref = y32.view(B, npatch + 1, D)[:, 1:].mean(1)
    lib.meanpool_fwd_(y16, y32, B, npatch)
    assert rel_err(y32.view(B, npatch + 1, D)[:, 0], ref) < 1e-6
    dout = torch.randn(B * (npatch + 1), D, generator=g)
    dy = lib.meanpool_bwd(dout.cuda(), B, npatch).cpu().view(B, npatch + 1, D)
    d3 = dout.view(B, npatch + 1, D)
    assert float(dy[:, 0].abs().max()) == 0.0
    assert rel_err(dy[:, 1:], d3[:, 1:] + d3[:, :1] / npatch) < 1e-6
    src = torch.randn(40, D, generator=g)
    idx = torch.randint(0, 40, (25,), generator=g)
    got = lib.gather_rows(src.cuda(), idx.cuda(), out_dtype=torch.bfloat16)
    assert torch.equal(got.cpu(), bf(src[idx]))
    dst = torch.zeros(40, D, device="cuda")
    lib.scatter_add_rows_(dst, idx.cuda(), src[:25].contiguous().cuda())
    assert rel_err(dst, torch.zeros(40, D).index_add_(0, idx, src[:25])) < 1e-6
    ws, H = 4, 2
    N = ws * ws + 1
    table = torch.randn((2 * ws - 1) ** 2 + 3, H, generator=g)
    rpi = O.relative_position_index(ws)
    bias = lib.relpos_bias_fwd(table.cuda(), rpi.cuda(), N, H, 24)
    ref_b = table[rpi.view(-1)].view(N, N, H).permute(2, 0, 1)
    assert torch.equal(bias.cpu()[:, :, :N], ref_b)
    db = torch.zeros(H, N, 24)
    db[:, :, :N] = torch.randn(H, N, N, generator=g)
    dt = torch.zeros_like(table).cuda()
    lib.relpos_bias_bwd(db.cuda(), rpi.cuda(), dt, N, H, 24)
    ref_dt = torch.zeros_like(table).index_add_(0, rpi.view(-1), db[:, :, :N].permute(1, 2, 0).reshape(-1, H))
    assert rel_err(dt, ref_dt) < 1e-5


# ------------------------------------------------------------------------------------------------ attention
def _attn_ref(q, k, v, scale, bias=None, kmask=None):
    s = (q * scale) @ k.transpose(-1, -2)
    if bias is not None:
        s = s + bias
    if kmask is not None:
        s = s + kmask[:, None, None, :]
    return torch.softmax(s, -1) @ v


@pytest.mark.parametrize("B,H,Lq,Lk,mode", [(3, 12, 197, 197, "vit"), (4, 12, 40, 40, "text"), (6, 12, 40, 197, "cross"),
                                            (2, 2, 17, 17, "vit"), (3, 2, 24, 17, "cross"), (2, 12, 577, 577, "vit")])
def test_attention_fwd_bwd(lib, B, H, Lq, Lk, mode):
    g = G(Lq * 7 + Lk)
    D = H * 64
    Bkv = B if mode != "cross" else max(1, B // 2)
    scale = 0.125
    if mode == "cross":
        q2 = bf(torch.randn(B * Lq, D, generator=g))
        kv2 = bf(torch.randn(Bkv * Lk, 2 * D, generator=g))
        qv, kvw, vvw = q2.cuda(), kv2.cuda()[:, :D], kv2.cuda()[:, D:]
        kv_index = torch.randint(0, Bkv, (B,), generator=g).to(torch.int32)
        kv_index[:Bkv] = torch.arange(Bkv, dtype=torch.int32)
        qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3)
        kf = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3)[kv_index.long()]
        vf = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3)[kv_index.long()]
    else:
        qkv = bf(torch.randn(B * Lq, 3 * D, generator=g))
        c = qkv.cuda()
        qv, kvw, vvw = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
        kv_index = None
        f = qkv.float().view(B, Lq, 3, H, 64).permute(2, 0, 3, 1, 4)
        qf, kf, vf = f[0], f[1], f[2]
    bias = kmask = None
    ld = (Lk + 7) // 8 * 8
    if mode == "vit":
        bias = torch.zeros(H, Lq, ld)
        bias[:, :, :Lk] = torch.randn(H, Lq, Lk, generator=g)
    if mode == "text":
        kmask = torch.zeros(B, Lk)
        kmask[1, Lk - 9:] = -10000.0
        kmask[2, 5:] = -10000.0
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (qf, kf, vf))
    bias_r = None if bias is None else bias[:, :, :Lk].clone().requires_grad_(True)
    ref = _attn_ref(qf, kf, vf, scale, bias_r, kmask)
    dout = bf(torch.randn(B * Lq, D, generator=g))
    ref.backward(dout.float().view(B, Lq, H, 64).permute(0, 2, 1, 3))
    out, lse = lib.attention_fwd(qv, kvw, vvw, B, H, Lq, Lk, scale, Bkv=Bkv, bias=None if bias is None else bias.cuda(),
                                 kmask=None if kmask is None else kmask.cuda(),
                                 kv_index=None if kv_index is None else kv_index.cuda())
    ref2 = ref.detach().permute(0, 2, 1, 3).reshape(B * Lq, D)
    assert float((out.float().cpu() - ref2).abs().max()) < 2e-2  # bf16 P and output rounding
    # backward
    if mode == "cross":
        dq = torch.empty(B * Lq, D, dtype=torch.bfloat16, device="cuda")
        dkv = torch.zeros(Bkv * Lk, 2 * D, dtype=torch.bfloat16, device="cuda")
        dk, dv = dkv[:, :D], dkv[:, D:]
        order = torch.argsort(kv_index.long(), stable=True).to(torch.int32)
        counts = torch.bincount(kv_index.long(), minlength=Bkv)
        offs = torch.zeros(Bkv + 1, dtype=torch.int32)
        offs[1:] = torch.cumsum(counts, 0).to(torch.int32)
        extra = dict(kv_index=kv_index.cuda(), kv_offsets=offs.cuda(), kv_samples=order.cuda())
    else:
        dqkv = torch.empty(B * Lq, 3 * D, dtype=torch.bfloat16, device="cuda")
        dq, dk, dv = dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:]
        extra = {}
    ds = torch.zeros(B, H, Lq, ld, dtype=torch.bfloat16, device="cuda") if mode == "vit" else None
    lib.attention_bwd(dout.cuda(), qv, kvw, vvw, out, lse, B, H, Lq, Lk, scale, dq, dk, dv, Bkv=Bkv,
                      bias=None if bias is None else bias.cuda(), kmask=None if kmask is None else kmask.cuda(),
                      ds_dump=ds, **extra)
    dq_ref = qf.grad.permute(0, 2, 1, 3).reshape(B * Lq, D)
    if mode == "cross":
        dk_full = kf.grad.permute(0, 2, 1, 3).reshape(B, Lk, D)
        dv_full = vf.grad.permute(0, 2, 1, 3).reshape(B, Lk, D)
        dk_ref = torch.zeros(Bkv, Lk, D).index_add_(0, kv_index.long(), dk_full).view(Bkv * Lk, D)
        dv_ref = torch.zeros(Bkv, Lk, D).index_add_(0, kv_index.long(), dv_full).view(Bkv * Lk, D)
    else:
        dk_ref = kf.grad.permute(0, 2, 1, 3).reshape(B * Lk, D)
        dv_ref = vf.grad.permute(0, 2, 1, 3).reshape(B * Lk, D)
    for name, got, want in (("dq", dq, dq_ref), ("dk", dk, dk_ref), ("dv", dv, dv_ref)):
        e = float((got.float().cpu() - want).abs().max())
        assert e < 2e-2 * max(1.0, float(want.abs().max())), (name, e, float(want.abs().max()))
    if ds is not None:
        dbias = lib.batch_sum_bf16(ds).cpu()[:, :, :Lk]
        e = float((dbias - bias_r.grad).abs().max())
        assert e < 2e-2 * max(1.0, float(bias_r.grad.abs().max())), e


@pytest.mark.parametrize("B,H,ws,with_table", [(3, 12, 14, True), (10, 12, 14, False), (2, 2, 4, True), (5, 3, 7, True),
                                               (1, 1, 12, True)])
def test_vit_attention_tcgen05_forward(lib, B, H, ws, with_table):
    """tcgen05 / TMEM forward (attention_tc.cu): relative-position bias gathered from the table in closed form
    (beit2.py:94-116,139-145) must equal softmax((q*scale) k^T + table[index]) v; also checked against the mma.sync
    kernel fed with the materialised bias, and lse against torch.logsumexp."""
    from xfm_b200.encoders import closed_form_rel_index
    g = G(ws * 100 + B)
    L, D = ws * ws + 1, H * 64
    qkv = bf(torch.randn(B * L, 3 * D, generator=g))
    c = qkv.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    f = qkv.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    table = bias = bias_dev = None
    if with_table:
        T = (2 * ws - 1) ** 2 + 3
        table = torch.randn(T, H, generator=g)
        idx = closed_form_rel_index(ws)
        bias = table[idx.view(-1)].view(L, L, H).permute(2, 0, 1).contiguous()  # beit2.py:139-145
        ld = (L + 7) // 8 * 8
        bias_dev = torch.zeros(H, L, ld)
        bias_dev[:, :, :L] = bias
        bias_dev = bias_dev.cuda()
    s = (f[0] * 0.125) @ f[1].transpose(-1, -2)
    if bias is not None:
        s = s + bias
    ref = (torch.softmax(s, -1) @ f[2]).permute(0, 2, 1, 3).reshape(B * L, D)
    lse_ref = torch.logsumexp(s, -1)
    kw = dict(bias=bias_dev, rel_table=None if table is None else table.cuda(), rel_window=ws if with_table else 0)
    out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, **kw)
    out2, lse2 = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, allow_tc=False, **kw)
    assert float((out.float().cpu() - ref).abs().max()) < 2e-2
    assert float((lse.cpu() - lse_ref).abs().max()) < 2e-3
    assert float((out.float() - out2.float()).abs().max()) < 2e-2
    assert float((lse - lse2).abs().max()) < 2e-3


@pytest.mark.parametrize("B,H,ws,with_table", [(3, 12, 14, True), (2, 2, 14, False), (2, 2, 4, True), (5, 3, 7, True),
                                               (2, 1, 12, True), (30, 12, 14, True)])
def test_vit_attention_tcgen05_fused_backward(lib, B, H, ws, with_table):
    """tcgen05 fused dQ / dK / dV kernel, with and without the bf16 dS dump, and the relative-position-table gradient reduced
    from that dump as the model does it, against torch autograd."""
    from xfm_b200.encoders import closed_form_rel_index
    g = G(ws * 1000 + B)
    L, D = ws * ws + 1, H * 64
    qkv = bf(torch.randn(B * L, 3 * D, generator=g) * 0.7)
    dout = bf(torch.randn(B * L, D, generator=g))
    f = qkv.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (f[0], f[1], f[2]))
    table = None
    s = (qf * 0.125) @ kf.transpose(-1, -2)
    if with_table:
        T = (2 * ws - 1) ** 2 + 3
        table = (torch.randn(T, H, generator=g)).requires_grad_(True)
        idx = closed_form_rel_index(ws)
        s = s + table[idx.view(-1)].view(L, L, H).permute(2, 0, 1)
    s.retain_grad()
    ref = torch.softmax(s, -1) @ vf
    ref.backward(dout.float().view(B, L, H, 64).permute(0, 2, 1, 3))
    want = torch.stack([qf.grad, kf.grad, vf.grad]).permute(1, 3, 0, 2, 4).reshape(B * L, 3 * D)
    c, do = qkv.cuda(), dout.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    tdev = None if table is None else table.detach().cuda()
    kw = dict(rel_table=tdev, rel_window=ws if with_table else 0)
    out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, **kw)
    dqkv = torch.full_like(c, float("nan"))
    n0 = lib.launch_count()
    lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], **kw)
    assert lib.launch_count() - n0 == 2      # row-delta kernel + one fused launch
    got = dqkv.float().cpu()
    assert torch.isfinite(got).all()
    scale = float(want.abs().max())
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        err = float((got[:, sl] - want[:, sl]).abs().max())
        assert err < 2.5e-2 * max(1.0, scale), (name, err, scale)
    # the same kernel with the bf16 dS dump
    ld = (L + 7) // 8 * 8
    ds = torch.zeros(B, H, L, ld, dtype=torch.bfloat16, device="cuda")
    dqkv2 = torch.full_like(c, float("nan"))
    lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv2[:, :D], dqkv2[:, D:2 * D], dqkv2[:, 2 * D:], ds_dump=ds, **kw)
    got2 = dqkv2.float().cpu()
    assert torch.isfinite(got2).all()
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        err = float((got2[:, sl] - want[:, sl]).abs().max())
        assert err < 2.5e-2 * max(1.0, scale), ("with dump: " + name, err, scale)
    err = float((ds[..., :L].float().cpu() - s.grad).abs().max())
    assert err < 1e-2 * max(1.0, float(s.grad.abs().max())), ("ds_dump", err)
    if table is not None:   # the table gradient from the dump, reduced as blocks.vit_block_bwd does
        dtab = torch.zeros_like(tdev)
        lib.relpos_bias_bwd(lib.batch_sum_bf16(ds), closed_form_rel_index(ws).cuda(), dtab, L, H, ld)
        err = float((dtab.cpu() - table.grad).abs().max())
        assert err < 2e-2 * max(1.0, float(table.grad.abs().max())), ("table grad", err, float(table.grad.abs().max()))


@pytest.mark.parametrize("B,H,with_table", [(2, 3, True), (1, 2, False), (5, 12, True), (32, 12, True)])
def test_vit_attention_tcgen05_forward_key_blocks(lib, B, H, with_table):
    """384 px (W = 24, 577 tokens) forward on tcgen05: one launch per block of 192 keys (block-normalised partial output +
    block lse) and a merge kernel, against an fp32 torch reference and against the mma.sync kernel (output and lse)."""
    from xfm_b200.encoders import closed_form_rel_index
    ws = 24
    g = G(ws * 77 + B)
    L, D = ws * ws + 1, H * 64
    qkv = bf(torch.randn(B * L, 3 * D, generator=g) * 0.7)
    ld = (L + 7) // 8 * 8
    table, bias = None, None
    c = qkv.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    f = c.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (f[0] * 0.125) @ f[1].transpose(-1, -2)
    if with_table:
        T = (2 * ws - 1) ** 2 + 3
        table = torch.randn(T, H, generator=g).cuda()
        dense = table[closed_form_rel_index(ws).view(-1).cuda()].view(L, L, H).permute(2, 0, 1)
        s = s + dense
        bias = torch.zeros(H, L, ld, device="cuda")
        bias[..., :L] = dense
    ref = (torch.softmax(s, -1) @ f[2]).permute(0, 2, 1, 3).reshape(B * L, D)
    lse_ref = torch.logsumexp(s, -1)
    n0 = lib.launch_count()
    out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bias, rel_table=table, rel_window=ws if with_table else 0)
    assert lib.launch_count() - n0 == 4      # three key-block launches + the merge
    out2, lse2 = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bias, allow_tc=False)
    assert torch.isfinite(out.float()).all()
    assert float((out.float() - ref).abs().max()) < 2e-2
    assert float((lse - lse_ref).abs().max()) < 2e-3
    assert float((out.float() - out2.float()).abs().max()) < 2e-2
    assert float((lse - lse2).abs().max()) < 2e-3


@pytest.mark.parametrize("B,H,with_table", [(2, 3, True), (1, 2, False), (5, 12, True)])
def test_vit_attention_tcgen05_backward_key_blocks(lib, B, H, with_table):
    """384 px (W = 24, 577 tokens): the fused tcgen05 backward runs one launch per block of 192 keys — dQ accumulated across the
    launches by TMA reduce-add, dK / dV rows and the dS columns written per block — against torch autograd.  The forward
    (and its lse) is the mma.sync kernel with the materialised bias."""
    from xfm_b200.encoders import closed_form_rel_index
    ws = 24
    g = G(ws * 1000 + B)
    L, D = ws * ws + 1, H * 64
    qkv = bf(torch.randn(B * L, 3 * D, generator=g) * 0.7)
    dout = bf(torch.randn(B * L, D, generator=g))
    f = qkv.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (f[0], f[1], f[2]))
    s = (qf * 0.125) @ kf.transpose(-1, -2)
    ld = (L + 7) // 8 * 8
    table, bias = None, None
    if with_table:
        T = (2 * ws - 1) ** 2 + 3
        table = torch.randn(T, H, generator=g)
        dense = table[closed_form_rel_index(ws).view(-1)].view(L, L, H).permute(2, 0, 1)
        s = s + dense
        bias = torch.zeros(H, L, ld)
        bias[..., :L] = dense
        bias = bias.cuda()
    s.retain_grad()
    ref = torch.softmax(s, -1) @ vf
    ref.backward(dout.float().view(B, L, H, 64).permute(0, 2, 1, 3))
    want = torch.stack([qf.grad, kf.grad, vf.grad]).permute(1, 3, 0, 2, 4).reshape(B * L, 3 * D)
    c, do = qkv.cuda(), dout.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bias)
    n0 = lib.launch_count()
    ds = torch.full((B, H, L, ld), float("nan"), dtype=torch.bfloat16, device="cuda")
    dqkv = torch.full_like(c, float("nan"))
    lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], bias=bias,
                      ds_dump=ds, rel_table=None if table is None else table.cuda(), rel_window=ws if with_table else 0)
    assert lib.launch_count() - n0 == 4      # row-delta kernel + three key-block launches (not the mma.sync pair)
    got = dqkv.float().cpu()
    assert torch.isfinite(got).all()
    scale = float(want.abs().max())
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        err = float((got[:, sl] - want[:, sl]).abs().max())
        assert err < 2.5e-2 * max(1.0, scale), (name, err, scale)
    dsf = ds.float().cpu()
    assert torch.isfinite(dsf).all() and float(dsf[..., L:].abs().max()) == 0.0      # padding columns are written as zeros
    err = float((dsf[..., :L] - s.grad).abs().max())
    assert err < 1e-2 * max(1.0, float(s.grad.abs().max())), ("ds_dump", err)


def _cross_case(B, Bkv, H, g, kv_index, Lk=197):
    Lq, D = 40, H * 64
    q2 = bf(torch.randn(B * Lq, D, generator=g))
    kv2 = bf(torch.randn(Bkv * Lk, 2 * D, generator=g))
    order = torch.argsort(kv_index.long(), stable=True).to(torch.int32)
    offs = torch.zeros(Bkv + 1, dtype=torch.int32)
    offs[1:] = torch.cumsum(torch.bincount(kv_index.long(), minlength=Bkv), 0).to(torch.int32)
    return Lq, Lk, D, q2, kv2, order, offs


@pytest.mark.parametrize("Lk_", [197, 577])
@pytest.mark.parametrize("B,Bkv,H,pattern", [(8, 2, 2, "even"), (24, 6, 12, "random"), (14, 2, 3, "big_groups"), (6, 6, 2, "identity")])
def test_cross_attention_tcgen05_forward(lib, B, Bkv, H, pattern, Lk_):
    """tcgen05 cross-attention (attention_xtc.cu): samples stacked per image (1..>GMAX samples per image) against torch and
    against the mma.sync kernel; with dropout the two kernels must produce the same mask (same (seed, index) hash).  577 image
    tokens (384 px): one launch per block of 192 keys + the merge of the block-normalised partials."""
    g = G(B * 31 + Bkv)
    if pattern == "even":
        kv_index = (torch.arange(B) % Bkv).to(torch.int32)
    elif pattern == "identity":
        kv_index = torch.arange(B, dtype=torch.int32)
    elif pattern == "big_groups":
        kv_index = torch.tensor([0] * 9 + [1] * 5, dtype=torch.int32)   # 9 > GMAX = 6: two chunks
    else:
        kv_index = torch.randint(0, Bkv, (B,), generator=g).to(torch.int32)
        kv_index[:Bkv] = torch.arange(Bkv, dtype=torch.int32)
    Lq, Lk, D, q2, kv2, order, offs = _cross_case(B, Bkv, H, g, kv_index, Lk=Lk_)
    qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3)
    kf = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3)[kv_index.long()]
    vf = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3)[kv_index.long()]
    s = (qf * 0.125) @ kf.transpose(-1, -2)
    ref = (torch.softmax(s, -1) @ vf).permute(0, 2, 1, 3).reshape(B * Lq, D)
    qd, kvd = q2.cuda(), kv2.cuda()
    kw = dict(Bkv=Bkv, kv_index=kv_index.cuda(), kv_offsets=offs.cuda(), kv_samples=order.cuda())
    n0 = lib.launch_count()
    out, lse = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, **kw)
    assert lib.launch_count() - n0 == (4 if Lk == 577 else 1)
    out2, lse2 = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, allow_tc=False, **kw)
    assert float((out.float().cpu() - ref).abs().max()) < 2e-2
    assert float((lse.cpu() - torch.logsumexp(s, -1)).abs().max()) < 2e-3
    assert float((out.float() - out2.float()).abs().max()) < 2e-2
    od, _ = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=0.2, dropout_seed=11, **kw)
    od2, _ = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=0.2, dropout_seed=11, allow_tc=False, **kw)
    assert float((od.float() - od2.float()).abs().max()) < 3e-2
    assert float((od.float() - out.float()).abs().max()) > 1e-2   # dropout did something


@pytest.mark.parametrize("B,Bkv,H,pattern", [(8, 2, 2, "even"), (24, 6, 12, "random"), (14, 2, 3, "big_groups"), (6, 6, 2, "identity")])
def test_cross_attention_tcgen05_backward(lib, B, Bkv, H, pattern):
    """tcgen05 cross-attention dQ / dK / dV against torch autograd (no dropout) and against the mma.sync kernels with the
    shared dropout mask (p = 0.2)."""
    g = G(B * 17 + Bkv)
    if pattern == "even":
        kv_index = (torch.arange(B) % Bkv).to(torch.int32)
    elif pattern == "identity":
        kv_index = torch.arange(B, dtype=torch.int32)
    elif pattern == "big_groups":
        kv_index = torch.tensor([0] * 9 + [1] * 5, dtype=torch.int32)
    else:
        kv_index = torch.randint(0, Bkv, (B,), generator=g).to(torch.int32)
        kv_index[:Bkv] = torch.arange(Bkv, dtype=torch.int32)
    Lq, Lk, D, q2, kv2, order, offs = _cross_case(B, Bkv, H, g, kv_index)
    dout = bf(torch.randn(B * Lq, D, generator=g))
    qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    kb = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    vb = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    s = (qf * 0.125) @ kb[kv_index.long()].transpose(-1, -2)
    ref = torch.softmax(s, -1) @ vb[kv_index.long()]
    ref.backward(dout.float().view(B, Lq, H, 64).permute(0, 2, 1, 3))
    want_dq = qf.grad.permute(0, 2, 1, 3).reshape(B * Lq, D)
    want_dk = kb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D)
    want_dv = vb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D)
    qd, kvd, do = q2.cuda(), kv2.cuda(), dout.cuda()
    kw = dict(Bkv=Bkv, kv_index=kv_index.cuda(), kv_offsets=offs.cuda(), kv_samples=order.cuda())

    def run(tc, p):
        out, lse = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=p, dropout_seed=9, allow_tc=tc, **kw)
        dq = torch.full_like(qd, float("nan"))
        dkv = torch.full_like(kvd, float("nan"))
        lib.attention_bwd(do, qd, kvd[:, :D], kvd[:, D:], out, lse, B, H, Lq, Lk, 0.125, dq, dkv[:, :D], dkv[:, D:],
                          dropout_p=p, dropout_seed=9, allow_tc=tc, **kw)
        return dq.float().cpu(), dkv[:, :D].float().cpu(), dkv[:, D:].float().cpu()

    dq, dk, dv = run(True, 0.0)
    for name, got, want in (("dq", dq, want_dq), ("dk", dk, want_dk), ("dv", dv, want_dv)):
        assert torch.isfinite(got).all(), name
        assert float((got - want).abs().max()) < 2.5e-2 * max(1.0, float(want.abs().max())), name
    a, b_ = run(True, 0.2), run(False, 0.2)
    for name, x, y in zip(("dq", "dk", "dv"), a, b_):
        assert torch.isfinite(x).all(), name
        assert float((x - y).abs().max()) < 3e-2 * max(1.0, float(y.abs().max())), name


@pytest.mark.parametrize("B,Bkv,H,pattern", [(8, 2, 2, "even"), (9, 3, 12, "random"), (14, 2, 3, "big_groups")])
def test_cross_attention_tcgen05_backward_key_blocks(lib, B, Bkv, H, pattern):
    """384 px: 40 text tokens attending to 577 image tokens.  The fused tcgen05 backward runs one launch per block of 192 keys
    (dQ accumulated across the launches by TMA reduce-add); the forward is the mma.sync kernel.  Against torch autograd
    (no dropout) and against the mma.sync backward with the shared dropout mask (p = 0.2: the key index inside the whole
    row feeds the hash)."""
    g = G(B * 19 + Bkv)
    if pattern == "even":
        kv_index = (torch.arange(B) % Bkv).to(torch.int32)
    elif pattern == "big_groups":
        kv_index = torch.tensor([0] * 9 + [1] * 5, dtype=torch.int32)
    else:
        kv_index = torch.randint(0, Bkv, (B,), generator=g).to(torch.int32)
        kv_index[:Bkv] = torch.arange(Bkv, dtype=torch.int32)
    Lq, Lk, D, q2, kv2, order, offs = _cross_case(B, Bkv, H, g, kv_index, Lk=577)
    dout = bf(torch.randn(B * Lq, D, generator=g))
    qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    kb = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    vb = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    s = (qf * 0.125) @ kb[kv_index.long()].transpose(-1, -2)
    ref = torch.softmax(s, -1) @ vb[kv_index.long()]
    ref.backward(dout.float().view(B, Lq, H, 64).permute(0, 2, 1, 3))
    want = (qf.grad.permute(0, 2, 1, 3).reshape(B * Lq, D), kb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D),
            vb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D))
    qd, kvd, do = q2.cuda(), kv2.cuda(), dout.cuda()
    kw = dict(Bkv=Bkv, kv_index=kv_index.cuda(), kv_offsets=offs.cuda(), kv_samples=order.cuda())

    def run(tc, p):
        out, lse = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=p, dropout_seed=9, allow_tc=tc, **kw)
        dq = torch.full_like(qd, float("nan"))
        dkv = torch.full_like(kvd, float("nan"))
        n0 = lib.launch_count()
        lib.attention_bwd(do, qd, kvd[:, :D], kvd[:, D:], out, lse, B, H, Lq, Lk, 0.125, dq, dkv[:, :D], dkv[:, D:],
                          dropout_p=p, dropout_seed=9, allow_tc=tc, **kw)
        return dq.float().cpu(), dkv[:, :D].float().cpu(), dkv[:, D:].float().cpu(), lib.launch_count() - n0

    dq, dk, dv, n = run(True, 0.0)
    assert n == 4      # row-delta kernel + three key-block launches
    for name, got, w in zip(("dq", "dk", "dv"), (dq, dk, dv), want):
        assert torch.isfinite(got).all(), name
        assert float((got - w).abs().max()) < 2.5e-2 * max(1.0, float(w.abs().max())), name
    a, b_ = run(True, 0.2), run(False, 0.2)
    assert b_[3] == 3  # row-delta + the two mma.sync kernels
    for name, x, y in zip(("dq", "dk", "dv"), a[:3], b_[:3]):
        assert torch.isfinite(x).all(), name
        assert float((x - y).abs().max()) < 3e-2 * max(1.0, float(y.abs().max())), name


@pytest.mark.parametrize("B,H,masked", [(3, 2, False), (7, 12, True), (96, 12, True), (1, 1, True), (11, 3, False)])
def test_self_attention_tcgen05(lib, B, H, masked):
    """tcgen05 text / fusion self-attention (attention_stc.cu): three 40-token samples packed per 128-row tile, additive key
    mask (xroberta.py:966-970), B not a multiple of 3, q/k/v as strided views of one qkv matrix.  Forward and the fused
    backward against torch autograd without dropout, and against the mma.sync kernels with the shared dropout mask."""
    g = G(B * 13 + H)
    L, D = 40, H * 64
    qkv = bf(torch.randn(B * L, 3 * D, generator=g))
    dout = bf(torch.randn(B * L, D, generator=g))
    km = None
    if masked:
        lens = torch.randint(3, L + 1, (B,), generator=g)
        km = torch.where(torch.arange(L)[None, :] < lens[:, None], 0.0, -10000.0)
    f = qkv.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (f[0], f[1], f[2]))
    s = (qf * 0.125) @ kf.transpose(-1, -2)
    if masked:
        s = s + km[:, None, None, :]
    ref = torch.softmax(s, -1) @ vf
    ref.backward(dout.float().view(B, L, H, 64).permute(0, 2, 1, 3))
    want = [t.grad.permute(0, 2, 1, 3).reshape(B * L, D) for t in (qf, kf, vf)]
    qd, do = qkv.cuda(), dout.cuda()
    kmd = None if km is None else km.cuda().contiguous()
    q, k, v = qd[:, :D], qd[:, D:2 * D], qd[:, 2 * D:]

    def run(tc, p):
        out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, kmask=kmd, dropout_p=p, dropout_seed=21, allow_tc=tc)
        dqkv = torch.full_like(qd, float("nan"))
        lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:],
                          kmask=kmd, dropout_p=p, dropout_seed=21, allow_tc=tc)
        return out.float().cpu(), lse.cpu(), dqkv.float().cpu()

    out, lse, dqkv = run(True, 0.0)
    assert float((out - ref.detach().permute(0, 2, 1, 3).reshape(B * L, D)).abs().max()) < 2e-2
    assert float((lse - torch.logsumexp(s.detach(), -1)).abs().max()) < 2e-3
    assert torch.isfinite(dqkv).all()
    for i, name in enumerate(("dq", "dk", "dv")):
        got, w = dqkv[:, i * D:(i + 1) * D], want[i]
        assert float((got - w).abs().max()) < 2.5e-2 * max(1.0, float(w.abs().max())), name
    a, b_ = run(True, 0.2), run(False, 0.2)
    assert float((a[0] - out).abs().max()) > 1e-2          # dropout did something
    assert float((a[0] - b_[0]).abs().max()) < 3e-2        # same mask in both kernel families
    assert float((a[1] - b_[1]).abs().max()) < 2e-3
    assert torch.isfinite(a[2]).all()
    assert float((a[2] - b_[2]).abs().max()) < 3e-2 * max(1.0, float(b_[2].abs().max()))


def test_attention_dropout_is_consistent(lib):
    """Same (seed, index) mask in forward and both backward kernels: check dQ/dK/dV against autograd through the
    forward's own (recovered) mask."""
    g = G(11)
    B, H, L, D = 2, 2, 24, 128
    qkv = bf(torch.randn(B * L, 3 * D, generator=g)).cuda()
    q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
    o0, _ = lib.attention_fwd(q, k, v, B, H, L, L, 0.125)
    o1, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, dropout_p=0.25, dropout_seed=5)
    o2, _ = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, dropout_p=0.25, dropout_seed=5)
    assert torch.equal(o1, o2) and not torch.equal(o0, o1)
    # recover the mask: with V = identity-like probes
    eye = torch.zeros(B * L, 3 * D, dtype=torch.bfloat16, device="cuda")
    eye[:, :2 * D] = qkv[:, :2 * D]
    for b in range(B):
        for h in range(H):
            eye[b * L:(b + 1) * L, 2 * D + h * 64:2 * D + h * 64 + L] = torch.eye(L, dtype=torch.bfloat16, device="cuda")
    pd, _ = lib.attention_fwd(eye[:, :D], eye[:, D:2 * D], eye[:, 2 * D:], B, H, L, L, 0.125, dropout_p=0.25, dropout_seed=5)
    pn, _ = lib.attention_fwd(eye[:, :D], eye[:, D:2 * D], eye[:, 2 * D:], B, H, L, L, 0.125)
    keep = (pd.float().view(B, L, H, 64)[..., :L] != 0) | (pn.float().view(B, L, H, 64)[..., :L] == 0)
    keep = keep.permute(0, 2, 1, 3).cpu()  # [B,H,Lq,Lk]
    frac = float(keep.float().mean())
    assert 0.6 < frac < 0.9
    f = qkv.float().cpu().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (f[0], f[1], f[2]))
    p = torch.softmax((qf * 0.125) @ kf.transpose(-1, -2), -1) * keep.float() / 0.75
    ref = p @ vf
    assert float((o1.float().cpu() - ref.detach().permute(0, 2, 1, 3).reshape(B * L, D)).abs().max()) < 3e-2
    dout = bf(torch.randn(B * L, D, generator=g))
    ref.backward(dout.float().view(B, L, H, 64).permute(0, 2, 1, 3))
    dqkv = torch.empty_like(qkv)
    lib.attention_bwd(dout.cuda(), q, k, v, o1, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:],
                      dropout_p=0.25, dropout_seed=5)
    want = torch.stack([qf.grad, kf.grad, vf.grad]).permute(1, 3, 0, 2, 4).reshape(B * L, 3 * D)
    assert float((dqkv.float().cpu() - want).abs().max()) < 3e-2 * max(1.0, float(want.abs().max()))


# ------------------------------------------------------------------------------------------------ losses
@pytest.mark.parametrize("R,V", [(37, 1000), (30, 50265)])
def test_cross_entropy(lib, R, V):
    g = G(V)
    ld = (V + 7) // 8 * 8
    logits = torch.zeros(R, ld)
    logits[:, :V] = torch.randn(R, V, generator=g) * 3
    labels = torch.randint(0, V, (R,), generator=g)
    labels[::5] = -100
    lr = logits[:, :V].clone().requires_grad_(True)
    ref = F.cross_entropy(lr, labels)
    (ref * 0.7).backward()
    lc = logits.cuda()
    loss, count, lse = lib.ce_fwd(lc, labels.cuda(), V)
    assert abs(float(loss) - float(ref)) < 1e-5 * max(1.0, abs(float(ref)))
    assert int(count) == int((labels >= 0).sum())
    d = lib.ce_bwd(lc, labels.cuda(), lse, count, torch.tensor([0.7], device="cuda"), V, ld)
    assert float(d[:, V:].abs().max() if ld > V else 0.0) == 0.0
    assert float((d[:, :V].float().cpu() - lr.grad).abs().max()) < 1e-2 * float(lr.grad.abs().max())


@pytest.mark.parametrize("use_idx", [False, True])
def test_itc_fused_loss_and_grads(lib, use_idx):
    g = G(21)
    n, E, off, ln = 48, 64, 16, 16  # rank 1 of 3
    fi = F.normalize(torch.randn(n, E, generator=g), dim=-1).requires_grad_(True)
    ft = F.normalize(torch.randn(n, E, generator=g), dim=-1).requires_grad_(True)
    temp = torch.tensor(0.07, requires_grad=True)
    idx = torch.randint(0, 9, (n,), generator=g) if use_idx else None
    ref = O.contrastive_loss(fi, ft, temp, idx_all=idx)
    ref.backward()
    loss, di, dt, dtemp = lib.itc_loss_fused(fi.detach().cuda(), ft.detach().cuda(), temp.detach().cuda().view(1), off, ln,
                                             None if idx is None else idx.cuda())
    assert abs(float(loss) - float(ref)) < 1e-5 * max(1.0, abs(float(ref)))
    assert rel_err(di, fi.grad[off:off + ln]) < 1e-4
    assert rel_err(dt, ft.grad[off:off + ln]) < 1e-4
    assert abs(float(dtemp) - float(temp.grad)) < 1e-4 * abs(float(temp.grad))


def test_itc_matches_reference_golden(lib, golden_dir):
    import os

    gold = torch.load(os.path.join(golden_dir, "itc_idx.pt"), weights_only=False)
    fi, ft, idx = gold["image_feat"], gold["text_feat"], gold["idx"]
    t = torch.tensor([gold["temp"]], device="cuda")
    n = fi.shape[0]
    l_idx, *_ = lib.itc_loss_fused(fi.cuda(), ft.cuda(), t, 0, n, idx.cuda())
    l_plain, *_ = lib.itc_loss_fused(fi.cuda(), ft.cuda(), t, 0, n, None)
    assert abs(float(l_idx) - gold["loss_idx"]) < 1e-5 and abs(float(l_plain) - gold["loss_plain"]) < 1e-5
    ineg, tneg, w_i2t, w_t2i = lib.hard_negatives(fi.cuda(), ft.cuda(), t, 3, idx=idx.cuda(), want_weights=True)
    torch.testing.assert_close(w_i2t.cpu(), gold["weights_i2t"], rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(w_t2i.cpu(), gold["weights_t2i"], rtol=1e-4, atol=1e-7)
    # draws land on admissible (non-zero weight) entries
    assert bool((gold["weights_t2i"][torch.arange(n), ineg.cpu()] > 0).all())
    assert bool((gold["weights_i2t"][torch.arange(n), tneg.cpu()] > 0).all())


def test_hard_negative_sampling_distribution(lib):
    g = G(31)
    B, E = 8, 32
    fi = F.normalize(torch.randn(B, E, generator=g), dim=-1)
    ft = F.normalize(torch.randn(B, E, generator=g), dim=-1)
    temp = torch.tensor(0.5)
    w_i2t, w_t2i = O.hard_negative_weights(fi, ft, temp)
    counts = torch.zeros(B, B)
    T = 4000
    for s in range(T):
        ineg, tneg, _, _ = lib.hard_negatives(fi.cuda(), ft.cuda(), temp.cuda().view(1), seed=s)
        counts[torch.arange(B), tneg.cpu()] += 1
    emp = counts / T
    want = w_i2t / w_i2t.sum(1, keepdim=True)
    assert float(emp.diagonal().max()) == 0.0
    assert float((emp - want).abs().max()) < 0.04


def test_vq_argmin_bit_exact(lib):
    g = G(41)
    B, Cd, K = 96, 32, 8192
    z = torch.randn(B, Cd, 14, 14, generator=g)
    code = F.normalize(torch.randn(K, Cd, generator=g), dim=-1)
    ref = O.quantizer_indices(z, code)
    amb = O.quantizer_ambiguous(z, code)
    zr = z.permute(0, 2, 3, 1).reshape(-1, Cd).contiguous()
    ids = lib.vq_argmin(zr.cuda(), code.cuda()).cpu()
    assert ids.dtype == torch.int64
    mism = ids != ref
    assert not bool((mism & ~amb).any()), f"{int((mism & ~amb).sum())} non-tie mismatches"
    assert int(mism.sum()) <= int(amb.sum())
    # exact ties must resolve to the first index: duplicate codes
    code2 = code.clone()
    code2[4000:4100] = code2[100:200]
    ids2 = lib.vq_argmin(zr.cuda(), code2.cuda()).cpu()
    assert not bool(((ids2 >= 4000) & (ids2 < 4100)).any())
    # empty / ragged row counts
    assert lib.vq_argmin(zr[:1].contiguous().cuda(), code.cuda()).cpu()[0] == ids[0]
    assert torch.equal(lib.vq_argmin(zr[:131].contiguous().cuda(), code.cuda()).cpu(), ids[:131])


def test_bbox_loss_and_region_pool_kernels_against_torch(lib):
    """xfm_bbox_loss (xfm.py:815-840 + box_ops.py) values and gradients against autograd of the oracle's restatement — with
    and without is_image, and the degenerate-box early-out; xfm_region_pool_fwd / _bwd (beit2.py:468-475) against torch."""
    L = lib
    g = torch.Generator().manual_seed(9)
    n = 37
    coord = torch.rand(n, 4, generator=g) * 0.5 + 0.2
    target = torch.rand(n, 4, generator=g) * 0.5 + 0.2
    is_image = (torch.rand(n, generator=g) < 0.3).float()
    for keep in (None, is_image):
        c = coord.clone().requires_grad_(True)
        lb, lg = O.bbox_loss(c, target, keep)
        gb, = torch.autograd.grad(lb, c, retain_graph=True)
        gg, = torch.autograd.grad(lg, c)
        mlb, mlg, db, dg = L.bbox_loss(coord.cuda(), target.cuda(), None if keep is None else keep.cuda())
        assert abs(float(mlb) - float(lb)) <= 1e-5 and abs(float(mlg) - float(lg)) <= 1e-5
        torch.testing.assert_close(db.cpu(), gb, rtol=1e-4, atol=1e-6)
        torch.testing.assert_close(dg.cpu(), gg, rtol=1e-3, atol=1e-5)
        up_b, up_g = torch.tensor([0.5], device="cuda"), torch.tensor([2.0], device="cuda")
        torch.testing.assert_close(L.axpby_scalars(db, up_b, dg, up_g).cpu(), 0.5 * gb + 2.0 * gg, rtol=1e-3, atol=1e-5)
    bad = coord.clone()
    bad[5, 2] = -0.1
    _, mlg, _, dg = L.bbox_loss(bad.cuda(), target.cuda(), None)
    assert float(mlg) == 0.0 and float(dg.abs().max()) == 0.0
    y = torch.sigmoid(coord)
    torch.testing.assert_close(L.sigmoid_fwd(coord.cuda()).cpu(), y, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(L.sigmoid_bwd(target.cuda(), y.cuda()).cpu(), target * y * (1 - y), rtol=1e-5, atol=1e-6)
    # region pooling
    n_img, N, D, bsz = 3, 17, 128, 7
    yv = torch.randn(n_img, N, D, generator=g)
    idx = torch.tensor([0, 0, 1, 2, 2, 2, 1])
    atts = (torch.rand(bsz, N, generator=g) < 0.5).long()
    atts[:, 0] = 1
    atts[:, 1] = 1
    yr = yv.clone().requires_grad_(True)
    x_bs = yr[:, 1:][idx]
    w = atts[:, 1:].unsqueeze(2)
    ref = torch.cat([(w * x_bs).sum(1, keepdim=True) / w.sum(1, keepdim=True), x_bs], 1)
    out, out16 = L.region_pool_fwd(yv.cuda(), idx.cuda(), atts.cuda())
    torch.testing.assert_close(out.cpu(), ref.detach(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(out16.float().cpu(), ref.detach(), rtol=1e-2, atol=1e-2)
    dout = torch.randn(bsz, N, D, generator=g)
    ref.backward(dout)
    dy = torch.zeros(n_img, N, D, device="cuda")
    L.region_pool_bwd_(dout.cuda(), idx.cuda(), atts.cuda(), dy)
    torch.testing.assert_close(dy.cpu(), yr.grad, rtol=1e-4, atol=1e-5)
