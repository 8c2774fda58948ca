"""Attention at 480 px (W = 30, 901 image tokens): the tcgen05 kernels in five key blocks (4 x 192 + 133) for ViT
self-attention and for 40-token cross-attention, and the streaming mma.sync kernels that serve every shape whose K / V
(or Q / dO) do not fit shared memory.  End to end: XFMForVQA at image_res 480 against the CPU oracle."""
import pytest
import torch

from oracle import dropout_mask as D
from oracle import xfm_oracle as O

pytestmark = pytest.mark.gpu

W30, L901 = 30, 901


@pytest.fixture(scope="module")
def lib():
    from xfm_b200 import lib as L

    L.lib()
    L.seed_salt_set(0)   # the dropout masks restated below depend on dropout_seed only
    return L


def G(seed=0):
    return torch.Generator(device="cpu").manual_seed(seed)


def bf(x):
    return x.to(torch.bfloat16)


def attn_keep_mask(B, H, Lq, Lk, seed, p):
    """attention.cu::drop_keep as [B, H, Lq, Lk]."""
    return torch.from_numpy(D.keep(seed, D.attention_index(B, H, Lq, Lk), p))


def kernel_names(fn):
    """Names of the CUDA kernels fn() launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _vit_case(B, H, with_table, seed, amp=0.7):
    from xfm_b200.encoders import closed_form_rel_index
    g = G(seed)
    L, D = L901, H * 64
    qkv = bf(torch.randn(B * L, 3 * D, generator=g) * amp)
    ld = (L + 7) // 8 * 8
    table = dense = bias = None
    if with_table:
        T = (2 * W30 - 1) ** 2 + 3
        table = torch.randn(T, H, generator=g)
        dense = table[closed_form_rel_index(W30).view(-1)].view(L, L, H).permute(2, 0, 1)
        bias = torch.zeros(H, L, ld)
        bias[..., :L] = dense
    return L, D, ld, qkv, table, dense, bias


# ------------------------------------------------------------------------------------------------ ViT self-attention
@pytest.mark.parametrize("B,H,with_table", [(1, 2, True), (1, 12, False), (5, 2, False), (5, 12, True), (24, 12, True)])
def test_vit_901_forward_key_blocks(lib, B, H, with_table):
    """Five launches (4 x 192 + 133 keys: the last block is the SHORTER one) + the merge, against fp32 torch and against the
    streaming mma.sync kernel fed with the materialised bias."""
    L, D, ld, qkv, table, dense, bias = _vit_case(B, H, with_table, 30 * 77 + B)
    c = qkv.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    f = c.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (f[0] * 0.125) @ f[1].transpose(-1, -2)
    if with_table:
        s = s + dense.cuda()
    ref = (torch.softmax(s, -1) @ f[2]).permute(0, 2, 1, 3).reshape(B * L, D)
    lse_ref = torch.logsumexp(s, -1)
    del s
    bd = None if bias is None else bias.cuda()
    n0 = lib.launch_count()
    out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bd, rel_table=None if table is None else table.cuda(),
                                 rel_window=W30 if with_table else 0)
    assert lib.launch_count() - n0 == 6      # five key-block launches + the merge
    out2, lse2 = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bd, allow_tc=False)
    assert torch.isfinite(out.float()).all()
    assert float((out.float() - ref).abs().max()) < 2e-2
    assert float((lse - lse_ref).abs().max()) < 2e-3
    assert float((out.float() - out2.float()).abs().max()) < 2e-2
    assert float((lse - lse2).abs().max()) < 2e-3


@pytest.mark.parametrize("B,H,with_table", [(2, 3, True), (1, 2, False), (5, 12, True)])
def test_vit_901_backward_key_blocks(lib, B, H, with_table):
    """Fused tcgen05 backward in five key blocks, with the dS dump, against torch autograd.  At W = 30 the table is staged
    without the CLS-row prefix (row 0 selects its constant), so query 0's dS row checks that branch."""
    L, D, ld, qkv, table, dense, bias = _vit_case(B, H, with_table, 30 * 1000 + B)
    g = G(B + 5)
    dout = bf(torch.randn(B * L, D, generator=g))
    f = qkv.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (f[0], f[1], f[2]))
    s = (qf * 0.125) @ kf.transpose(-1, -2)
    if with_table:
        s = s + dense
    s.retain_grad()
    ref = torch.softmax(s, -1) @ vf
    ref.backward(dout.float().view(B, L, H, 64).permute(0, 2, 1, 3))
    want = torch.stack([qf.grad, kf.grad, vf.grad]).permute(1, 3, 0, 2, 4).reshape(B * L, 3 * D)
    c, do = qkv.cuda(), dout.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    bd = None if bias is None else bias.cuda()
    out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bd)
    ds = torch.full((B, H, L, ld), float("nan"), dtype=torch.bfloat16, device="cuda")
    dqkv = torch.full_like(c, float("nan"))
    n0 = lib.launch_count()
    lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], bias=bd,
                      ds_dump=ds, rel_table=None if table is None else table.cuda(), rel_window=W30 if with_table else 0)
    assert lib.launch_count() - n0 == 6      # row-delta kernel + five key-block launches
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


# ------------------------------------------------------------------------------------------------ cross-attention 40 x 901
def _kv_index(pattern, B, Bkv, g):
    if pattern == "even":
        return (torch.arange(B) % Bkv).to(torch.int32)
    if pattern == "identity":
        return torch.arange(B, dtype=torch.int32)
    if pattern == "big_groups":
        return torch.tensor([0] * 9 + [1] * 5, dtype=torch.int32)   # 9 > GMAX: two chunks
    kv_index = torch.randint(0, Bkv, (B,), generator=g).to(torch.int32)
    kv_index[:Bkv] = torch.arange(Bkv, dtype=torch.int32)
    return kv_index


def _cross(B, Bkv, H, pattern, seed, Lq=40, Lk=L901):
    g = G(seed)
    kv_index = _kv_index(pattern, B, Bkv, g)
    D = H * 64
    q2 = bf(torch.randn(B * Lq, D, generator=g))
    kv2 = bf(torch.randn(Bkv * Lk, 2 * D, generator=g))
    dout = bf(torch.randn(B * Lq, D, generator=g))
    order = torch.argsort(kv_index.long(), stable=True).to(torch.int32)
    offs = torch.zeros(Bkv + 1, dtype=torch.int32)
    offs[1:] = torch.cumsum(torch.bincount(kv_index.long(), minlength=Bkv), 0).to(torch.int32)
    kw = dict(Bkv=Bkv, kv_index=kv_index.cuda(), kv_offsets=offs.cuda(), kv_samples=order.cuda())
    return kv_index, D, q2, kv2, dout, kw


CROSS = [(8, 2, 2, "even"), (24, 6, 12, "random"), (14, 2, 3, "big_groups"), (6, 6, 2, "identity")]


@pytest.mark.parametrize("B,Bkv,H,pattern", CROSS)
def test_cross_901_forward_key_blocks(lib, B, Bkv, H, pattern):
    Lq, Lk = 40, L901
    kv_index, D, q2, kv2, _, kw = _cross(B, Bkv, H, pattern, B * 31 + Bkv)
    qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3)
    kf = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3)[kv_index.long()]
    vf = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3)[kv_index.long()]
    s = (qf * 0.125) @ kf.transpose(-1, -2)
    ref = (torch.softmax(s, -1) @ vf).permute(0, 2, 1, 3).reshape(B * Lq, D)
    qd, kvd = q2.cuda(), kv2.cuda()
    n0 = lib.launch_count()
    out, lse = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, **kw)
    assert lib.launch_count() - n0 == 6      # five key-block launches + the merge
    out2, _ = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, allow_tc=False, **kw)
    assert float((out.float().cpu() - ref).abs().max()) < 2e-2
    assert float((lse.cpu() - torch.logsumexp(s, -1)).abs().max()) < 2e-3
    assert float((out.float() - out2.float()).abs().max()) < 2e-2
    od, _ = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=0.2, dropout_seed=11, **kw)
    od2, _ = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=0.2, dropout_seed=11, allow_tc=False,
                               **kw)
    assert float((od.float() - od2.float()).abs().max()) < 3e-2     # same mask across the five blocks
    assert float((od.float() - out.float()).abs().max()) > 1e-2     # dropout did something


@pytest.mark.parametrize("B,Bkv,H,pattern", CROSS)
def test_cross_901_backward_key_blocks(lib, B, Bkv, H, pattern):
    Lq, Lk = 40, L901
    kv_index, D, q2, kv2, dout, kw = _cross(B, Bkv, H, pattern, B * 19 + Bkv)
    qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    kb = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    vb = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    s = (qf * 0.125) @ kb[kv_index.long()].transpose(-1, -2)
    ref = torch.softmax(s, -1) @ vb[kv_index.long()]
    ref.backward(dout.float().view(B, Lq, H, 64).permute(0, 2, 1, 3))
    want = (qf.grad.permute(0, 2, 1, 3).reshape(B * Lq, D), kb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D),
            vb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D))
    qd, kvd, do = q2.cuda(), kv2.cuda(), dout.cuda()

    def run(tc, p):
        out, lse = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, dropout_p=p, dropout_seed=9, allow_tc=tc,
                                     **kw)
        dq = torch.full_like(qd, float("nan"))
        dkv = torch.full_like(kvd, float("nan"))
        n0 = lib.launch_count()
        lib.attention_bwd(do, qd, kvd[:, :D], kvd[:, D:], out, lse, B, H, Lq, Lk, 0.125, dq, dkv[:, :D], dkv[:, D:],
                          dropout_p=p, dropout_seed=9, allow_tc=tc, **kw)
        return dq.float().cpu(), dkv[:, :D].float().cpu(), dkv[:, D:].float().cpu(), lib.launch_count() - n0

    dq, dk, dv, n = run(True, 0.0)
    assert n == 6      # row-delta kernel + five key-block launches
    for name, got, w in zip(("dq", "dk", "dv"), (dq, dk, dv), want):
        assert torch.isfinite(got).all(), name
        assert float((got - w).abs().max()) < 2.5e-2 * max(1.0, float(w.abs().max())), name
    a, b_ = run(True, 0.2), run(False, 0.2)
    assert b_[3] == 3  # row-delta + the two mma.sync kernels
    for name, x, y in zip(("dq", "dk", "dv"), a[:3], b_[:3]):
        assert torch.isfinite(x).all(), name
        assert float((x - y).abs().max()) < 3e-2 * max(1.0, float(y.abs().max())), name


# ------------------------------------------------------------------------------------------------ streaming mma.sync kernels
def _torch_attn(qf, kf, vf, scale, addend=None, keep=None, p=0.0):
    s = (qf * scale) @ kf.transpose(-1, -2)
    if addend is not None:
        s = s + addend
    s.retain_grad()
    pr = torch.softmax(s, -1)
    if keep is not None:
        pr = pr * keep.float() / (1.0 - p)
    return s, pr @ vf


def _check(got, want, tol, name):
    assert torch.isfinite(got).all(), name
    err = float((got - want).abs().max())
    assert err < tol * max(1.0, float(want.abs().max())), (name, err, float(want.abs().max()))


def test_streaming_cross_12_queries_kmask(lib):
    """Lq = 12 cross-attention over 901 image tokens with a key mask (no tcgen05 path for Lq != 40): forward and dQ stream
    K / V through shared memory, dK / dV stay resident.  Against torch autograd."""
    B, Bkv, H, Lq, Lk = 6, 3, 12, 12, L901
    kv_index, D, q2, kv2, dout, kw = _cross(B, Bkv, H, "random", 123, Lq=Lq)
    g = G(7)
    km = torch.where(torch.rand(B, Lk, generator=g) < 0.2, -10000.0, 0.0)
    qf = q2.float().view(B, Lq, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    kb = kv2.float()[:, :D].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    vb = kv2.float()[:, D:].reshape(Bkv, Lk, H, 64).permute(0, 2, 1, 3).clone().requires_grad_(True)
    _, ref = _torch_attn(qf, kb[kv_index.long()], vb[kv_index.long()], 0.125, km[:, None, None, :])
    ref.backward(dout.float().view(B, Lq, H, 64).permute(0, 2, 1, 3))
    qd, kvd, do, kmd = q2.cuda(), kv2.cuda(), dout.cuda(), km.cuda()
    res = {}

    def run():
        out, lse = lib.attention_fwd(qd, kvd[:, :D], kvd[:, D:], B, H, Lq, Lk, 0.125, kmask=kmd, **kw)
        dq, dkv = torch.full_like(qd, float("nan")), torch.full_like(kvd, float("nan"))
        lib.attention_bwd(do, qd, kvd[:, :D], kvd[:, D:], out, lse, B, H, Lq, Lk, 0.125, dq, dkv[:, :D], dkv[:, D:], kmask=kmd,
                          **kw)
        res.update(out=out, lse=lse, dq=dq, dkv=dkv)

    names = kernel_names(run)
    assert any("attn_fwd_kernel<4, true>" in n for n in names), names
    assert any("attn_bwd_dq_kernel<4, true>" in n for n in names), names
    assert any("attn_bwd_dkv_kernel<8, false>" in n for n in names), names
    _check(res["out"].float().cpu(), ref.detach().permute(0, 2, 1, 3).reshape(B * Lq, D), 2e-2, "out")
    _check(res["dq"].float().cpu(), qf.grad.permute(0, 2, 1, 3).reshape(B * Lq, D), 2.5e-2, "dq")
    _check(res["dkv"][:, :D].float().cpu(), kb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D), 2.5e-2, "dk")
    _check(res["dkv"][:, D:].float().cpu(), vb.grad.permute(0, 2, 1, 3).reshape(Bkv * Lk, D), 2.5e-2, "dv")


@pytest.mark.parametrize("L,p", [(L901, 0.2), (1025, 0.0)])
def test_streaming_self_attention_bias_dropout_ds_dump(lib, L, p):
    """Self-attention that no resident kernel holds: 901 tokens with a dense bias, dropout (the mask restated from the hash)
    and the dS dump; 1025 tokens (W = 32, which no tcgen05 kernel takes) with a bias.  All three kernels stream."""
    B, H = 2, 2
    D = H * 64
    g = G(L + 3)
    qkv = bf(torch.randn(B * L, 3 * D, generator=g) * 0.7)
    dout = bf(torch.randn(B * L, D, generator=g))
    ld = (L + 7) // 8 * 8
    dense = torch.randn(H, L, L, generator=g)
    bias = torch.zeros(H, L, ld)
    bias[..., :L] = dense
    keep = attn_keep_mask(B, H, L, L, 17, p) if p > 0 else None
    f = qkv.float().view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    qf, kf, vf = (t.clone().requires_grad_(True) for t in (f[0], f[1], f[2]))
    s, ref = _torch_attn(qf, kf, vf, 0.125, dense, keep, p)
    ref.backward(dout.float().view(B, L, H, 64).permute(0, 2, 1, 3))
    c, do, bd = qkv.cuda(), dout.cuda(), bias.cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    res = {}

    def run():
        out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, bias=bd, dropout_p=p, dropout_seed=17)
        ds = torch.full((B, H, L, ld), float("nan"), dtype=torch.bfloat16, device="cuda")
        ds[..., L:] = 0          # the mma.sync kernels leave the padding columns to the caller
        dqkv = torch.full_like(c, float("nan"))
        lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], bias=bd,
                          ds_dump=ds, dropout_p=p, dropout_seed=17)
        res.update(out=out, lse=lse, ds=ds, dqkv=dqkv)

    names = kernel_names(run)
    for kname in ("attn_fwd_kernel<8, true>", "attn_bwd_dq_kernel<8, true>", "attn_bwd_dkv_kernel<8, true>"):
        assert any(kname in n for n in names), (kname, names)
    _check(res["out"].float().cpu(), ref.detach().permute(0, 2, 1, 3).reshape(B * L, D), 2e-2, "out")
    assert float((res["lse"].cpu() - torch.logsumexp(s.detach(), -1)).abs().max()) < 2e-3
    want = torch.stack([qf.grad, kf.grad, vf.grad]).permute(1, 3, 0, 2, 4).reshape(B * L, 3 * D)
    got = res["dqkv"].float().cpu()
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        _check(got[:, sl], want[:, sl], 2.5e-2, name)
    _check(res["ds"].float().cpu()[..., :L], s.grad, 1e-2, "ds_dump")


def test_resident_shapes_keep_resident_kernels(lib):
    """577 tokens with allow_tc=False fit the resident kernels: they, not the streaming variants, run."""
    B, H, L = 1, 2, 577
    D = H * 64
    c = bf(torch.randn(B * L, 3 * D, generator=G(1))).cuda()
    q, k, v = c[:, :D], c[:, D:2 * D], c[:, 2 * D:]
    do = bf(torch.randn(B * L, D, generator=G(2))).cuda()

    def run():
        out, lse = lib.attention_fwd(q, k, v, B, H, L, L, 0.125, allow_tc=False)
        dqkv = torch.empty_like(c)
        lib.attention_bwd(do, q, k, v, out, lse, B, H, L, L, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], allow_tc=False)

    names = kernel_names(run)
    for kname in ("attn_fwd_kernel<8, false>", "attn_bwd_dq_kernel<8, false>", "attn_bwd_dkv_kernel<8, false>"):
        assert any(kname in n for n in names), (kname, names)
    assert not any(", true>" in n for n in names), names


# ------------------------------------------------------------------------------------------------ end to end, 480 px
def _maxabs(a, b):
    return float((a.float().cpu() - b.float().cpu()).abs().max())


@pytest.mark.parametrize("Lq", [40, 12])
def test_vqa_480px_base_width_against_oracle(lib, Lq):
    """XFMForVQA at the XFM-base widths with image_res 480 (901 image tokens; 2 layers per stack), train mode off: loss,
    per-answer losses and gradients — vision qkv and the relative-position table included — against the CPU oracle.
    40-token questions take the tcgen05 cross-attention in five key blocks, 12-token ones the streaming fallback."""
    from xfm_b200.model_generation import XFMForVQA
    import types
    cfg = O.base_config(image_res=480, vision_depth=2, text_layers=2, fusion_layers=2, dec_layers=2, use_bbox=False)
    sd = O.make_state_dict(cfg, 0)
    for v in sd.values():
        if v.dtype.is_floating_point:
            v.requires_grad_(True)
    b = O.make_vqa_batch(cfg, B=4, L=Lq, La=8, n_cand=9, seed=17)
    col = {}
    ref = O.vqa_train_loss(b["image"], b["q_ids"], b["q_atts"], b["a_ids"], b["a_atts"], b["k"], b["weights"], sd, cfg,
                           collect=col)
    ref.backward()
    model = XFMForVQA(dict(cfg, num_dec_layers=2, pad_token_id=cfg["pad_id"]), init=lambda n, s: O.make_tensor(n, s, 0),
                      device="cuda").eval()
    c = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in b.items()}
    q = types.SimpleNamespace(input_ids=c["q_ids"], attention_mask=c["q_atts"])
    a = types.SimpleNamespace(input_ids=c["a_ids"], attention_mask=c["a_atts"])
    loss = model(c["image"], q, a, k=b["k"], weights=c["weights"], train=True)
    assert _maxabs(model.last_answer_loss, col["answer_loss"].detach()) <= 2e-3 * float(col["answer_loss"].abs().max())
    assert abs(float(loss) - float(ref)) <= 1e-3 * abs(float(ref)), (float(loss), float(ref))
    loss.backward()
    params = dict(model.named_parameters())
    for n in ["text_decoder.roberta.encoder.layer.0.crossattention.self.value.weight",
              "fusion_encoder.roberta.encoder.layer.0.crossattention.self.key.weight",
              "fusion_encoder.roberta.encoder.layer.1.output.dense.weight",
              "text_encoder.roberta.encoder.layer.0.attention.self.query.weight",
              "vision_encoder.blocks.0.attn.qkv.weight",
              "vision_encoder.blocks.0.attn.relative_position_bias_table",
              "vision_encoder.blocks.1.attn.relative_position_bias_table"]:
        mine, want = params[n].grad, sd[n].grad
        assert mine is not None and want is not None, n
        assert _maxabs(mine, want) <= 6e-2 * max(float(want.abs().max()), 1e-8), n
