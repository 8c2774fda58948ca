"""Encoders and heads of the XFM hot path as explicit forward / backward schedules over the C-ABI kernels.

    VisionEncoder   models/beit2.py:423-475 (forward_avgpool) and, with layerscale/relbias off and an absolute position
                    embedding, the VQ-KD tokenizer encoder models/vqkd_vit.py:373-408
    RobertaStack    models/xroberta.py:104-137 (embeddings) + :484-589 (12 post-LN layers, optional cross-attention)
    heads           get_features (xfm.py:614-621), itm_head (xfm.py:115-121), RobertaLMHead (xroberta.py:1313-1333)

There is no autograd in here: every *_fwd returns a state object, every *_bwd consumes it and accumulates parameter
gradients into the flat gradient buffer (params.FlatParams.G).  xfm.py wraps these in torch.autograd.Function so the
reference's call sites (loss.backward()) keep working.
"""
import math

import torch

from . import blocks as BK
from . import lib as L


class State:
    pass


def _f32(t):
    return t if t.dtype == torch.float32 else t.float()


def closed_form_rel_index(ws):
    """idx(i, j) of beit2.py:104-114 as arithmetic: what attention_tc.cu evaluates per score element."""
    T = (2 * ws - 1) ** 2 + 3
    n = ws * ws + 1
    t = torch.arange(n) - 1
    r, c = torch.div(t, ws, rounding_mode="floor"), t % ws
    idx = (r[:, None] - r[None, :] + ws - 1) * (2 * ws - 1) + (c[:, None] - c[None, :] + ws - 1)
    idx[0, :] = T - 3
    idx[:, 0] = T - 2
    idx[0, 0] = T - 1
    return idx.to(torch.int64)


# =====================================================================================================
# parameter layout
# =====================================================================================================
def add_vision(fp, cfg, init, prefix="vision_encoder.", layerscale=True, relbias=True, abs_pos=False, mask_token=True,
               trainable=True):
    D, Fv, Hh, P = cfg["vision_width"], cfg["vision_mlp"], cfg["vision_heads"], cfg["patch_size"]
    ws = cfg["image_res"] // P

    def add(name, shape, value=None, train=trainable):
        fp.add(prefix + name, shape, init=init(prefix + name, shape) if value is None else value, trainable=train)

    add("cls_token", (1, 1, D))
    if mask_token:
        add("mask_token", (1, 1, D))
    if abs_pos:
        add("pos_embed", (1, ws * ws + 1, D))
    add("patch_embed.proj.weight", (D, 3, P, P))
    add("patch_embed.proj.bias", (D,))
    for i in range(cfg["vision_depth"]):
        b = f"blocks.{i}."
        if layerscale:
            add(b + "gamma_1", (D,))
            add(b + "gamma_2", (D,))
        add(b + "norm1.weight", (D,))
        add(b + "norm1.bias", (D,))
        # q_bias | zeros | v_bias back to back = the fused qkv bias of beit2.py:128-132 (K has no bias)
        add(b + "attn.q_bias", (D,))
        add(b + "attn._k_bias", (D,), value=torch.zeros(D), train=False)
        add(b + "attn.v_bias", (D,))
        if relbias:
            add(b + "attn.relative_position_bias_table", ((2 * ws - 1) ** 2 + 3, Hh))
        add(b + "attn.qkv.weight", (3 * D, D))
        add(b + "attn.proj.weight", (D, D))
        add(b + "attn.proj.bias", (D,))
        add(b + "norm2.weight", (D,))
        add(b + "norm2.bias", (D,))
        add(b + "mlp.fc1.weight", (Fv, D))
        add(b + "mlp.fc1.bias", (Fv,))
        add(b + "mlp.fc2.weight", (D, Fv))
        add(b + "mlp.fc2.bias", (D,))
    add("fc_norm.weight", (D,))
    add("fc_norm.bias", (D,))


class TextNames:
    """Parameter naming of a text stack: models/xroberta.py (RobertaForMaskedLM: roberta.*, lm_head.*, lm_cap_head.*) or
    models/xbert.py (BertForMaskedLM: bert.*, cls.predictions.*, xbert.py:663-707,1523-1540).  The arithmetic of the two is
    the same post-LN layer; they differ in the embeddings (BERT: absolute position ids, xbert.py:167-221) and in where the
    1/sqrt(d) sits (xbert.py:296-301,329-330: on q when config.fp16, else on the scores) — at head_dim 64 the factor is
    0.125, a power of two, so both orders give bit-identical results and one kernel serves both."""

    def __init__(self, arch="roberta"):
        assert arch in ("roberta", "bert"), arch
        self.arch = arch
        self.stem = arch + "."

    def head(self, head="lm_head"):
        if self.arch == "roberta":
            h = head + "."
            return dict(bias=h + "bias", dense_w=h + "dense.weight", dense_b=h + "dense.bias", ln_w=h + "layer_norm.weight",
                        ln_b=h + "layer_norm.bias", dec_w=h + "decoder.weight", dec_b=h + "decoder.bias")
        h = "cls.predictions."
        return dict(bias=h + "bias", dense_w=h + "transform.dense.weight", dense_b=h + "transform.dense.bias",
                    ln_w=h + "transform.LayerNorm.weight", ln_b=h + "transform.LayerNorm.bias", dec_w=h + "decoder.weight",
                    dec_b=h + "decoder.bias")


def add_roberta(fp, cfg, init, prefix, layers, cross, enc_width, heads=("lm_head", "lm_cap_head"), arch="roberta"):
    H, Ff, V = cfg["hidden"], cfg["ffn"], cfg["vocab_size"]
    names = TextNames(arch)
    if arch == "bert":
        heads = ("lm_head",) if heads else ()   # BertForMaskedLM has the one prediction head

    def add(name, shape):
        fp.add(prefix + name, shape, init=init(prefix + name, shape))

    e = names.stem + "embeddings."
    add(e + "word_embeddings.weight", (V, H))
    add(e + "position_embeddings.weight", (cfg["max_pos"], H))
    add(e + "token_type_embeddings.weight", (cfg["type_vocab"], H))
    add(e + "LayerNorm.weight", (H,))
    add(e + "LayerNorm.bias", (H,))
    for i in range(layers):
        l = f"{names.stem}encoder.layer.{i}."
        a = l + "attention."
        # query | key | value back to back: one fused [3H, H] operand (xroberta.py:170-176 keeps three Linears)
        for n in ("query", "key", "value"):
            add(a + f"self.{n}.weight", (H, H))
        for n in ("query", "key", "value"):
            add(a + f"self.{n}.bias", (H,))
        add(a + "output.dense.weight", (H, H))
        add(a + "output.dense.bias", (H,))
        add(a + "output.LayerNorm.weight", (H,))
        add(a + "output.LayerNorm.bias", (H,))
        if cross:
            c = l + "crossattention."
            add(c + "self.query.weight", (H, H))
            add(c + "self.query.bias", (H,))
            add(c + "self.key.weight", (H, enc_width))
            add(c + "self.value.weight", (H, enc_width))
            add(c + "self.key.bias", (H,))
            add(c + "self.value.bias", (H,))
            add(c + "output.dense.weight", (H, H))
            add(c + "output.dense.bias", (H,))
            add(c + "output.LayerNorm.weight", (H,))
            add(c + "output.LayerNorm.bias", (H,))
        add(l + "intermediate.dense.weight", (Ff, H))
        add(l + "intermediate.dense.bias", (Ff,))
        add(l + "output.dense.weight", (H, Ff))
        add(l + "output.dense.bias", (H,))
        add(l + "output.LayerNorm.weight", (H,))
        add(l + "output.LayerNorm.bias", (H,))
    for head in heads:
        n = names.head(head)
        add(n["bias"], (V,))
        add(n["dense_w"], (H, H))
        add(n["dense_b"], (H,))
        add(n["ln_w"], (H,))
        add(n["ln_b"], (H,))
        if head == "lm_cap_head":  # untied decoder; lm_head.decoder.weight IS the word embedding (xroberta.py:1209-1210)
            add(n["dec_w"], (V, H))


def add_mlp_head(fp, init, name, din, dout):
    """build_mlp (xfm.py:115-121): Linear(din, 2 din) - LayerNorm - GELU - Linear(2 din, dout)."""
    for n, shape in ((".0.weight", (2 * din, din)), (".0.bias", (2 * din,)), (".1.weight", (2 * din,)),
                     (".1.bias", (2 * din,)), (".3.weight", (dout, 2 * din)), (".3.bias", (dout,))):
        fp.add(name + n, shape, init=init(name + n, shape))


# =====================================================================================================
# vision encoder
# =====================================================================================================
class VisionEncoder:
    def __init__(self, fp, cfg, prefix="vision_encoder.", layerscale=True, relbias=True, abs_pos=False, rel_index=None):
        self.fp, self.cfg, self.prefix = fp, cfg, prefix
        self.layerscale, self.relbias, self.abs_pos = layerscale, relbias, abs_pos
        self.D, self.H, self.P = cfg["vision_width"], cfg["vision_heads"], cfg["patch_size"]
        self.depth = cfg["vision_depth"]
        self.np = (cfg["image_res"] // self.P) ** 2
        self.N = self.np + 1
        self.eps = cfg["vision_ln_eps"] if prefix == "vision_encoder." else 1e-6  # model_vqkd.py:245
        self.rel_index = rel_index  # int64 [N, N] device tensor
        # The tcgen05 attention kernel gathers the bias through the closed form of beit2.py:104-114; use it only when the
        # buffer really is that index (a checkpoint could in principle carry another one).
        self.ws = cfg["image_res"] // self.P
        self.rel_closed_form = bool(relbias and rel_index is not None and
                                    torch.equal(rel_index.cpu(), closed_form_rel_index(self.ws)))
        self.bias_ld = (self.N + 7) // 8 * 8
        self.drop_path = [float(x) for x in torch.linspace(0, cfg["drop_path_rate"], self.depth)] if layerscale else \
            [0.0] * self.depth  # beit2.py:309; the frozen tokenizer runs in eval mode
        self.w = None
        self.collect = None  # tests: list receiving a f32 copy of every block output

    def refresh(self):
        fp, p, D = self.fp, self.prefix, self.D
        self.w, self.gmap = [], []
        for i in range(self.depth):
            b = f"{p}blocks.{i}."
            w = dict(n1w=fp.view32(b + "norm1.weight"), n1b=fp.view32(b + "norm1.bias"),
                     qkv_w16=fp.view16(b + "attn.qkv.weight"),
                     qkv_b=fp.span32(b + "attn.q_bias", b + "attn.v_bias", (3 * D,)),
                     proj_w16=fp.view16(b + "attn.proj.weight"), proj_b=fp.view32(b + "attn.proj.bias"),
                     n2w=fp.view32(b + "norm2.weight"), n2b=fp.view32(b + "norm2.bias"),
                     fc1_w16=fp.view16(b + "mlp.fc1.weight"), fc1_b=fp.view32(b + "mlp.fc1.bias"),
                     fc2_w16=fp.view16(b + "mlp.fc2.weight"), fc2_b=fp.view32(b + "mlp.fc2.bias"))
            gm = dict(n1w=b + "norm1.weight", n1b=b + "norm1.bias", qkv_w=b + "attn.qkv.weight", q_bias=b + "attn.q_bias",
                      v_bias=b + "attn.v_bias", proj_w=b + "attn.proj.weight", proj_b=b + "attn.proj.bias",
                      n2w=b + "norm2.weight", n2b=b + "norm2.bias", fc1_w=b + "mlp.fc1.weight", fc1_b=b + "mlp.fc1.bias",
                      fc2_w=b + "mlp.fc2.weight", fc2_b=b + "mlp.fc2.bias")
            if self.layerscale:
                w["g1"], w["g2"] = fp.view32(b + "gamma_1"), fp.view32(b + "gamma_2")
                gm["g1"], gm["g2"] = b + "gamma_1", b + "gamma_2"
            if self.relbias:
                w["rel_table"] = fp.view32(b + "attn.relative_position_bias_table")
                gm["rel_table"] = b + "attn.relative_position_bias_table"
            self.w.append(w)
            self.gmap.append(gm)
        self.pe_w16 = fp.view16(p + "patch_embed.proj.weight").view(D, -1)
        self.pe_b = fp.view32(p + "patch_embed.proj.bias")
        self.cls = fp.view32(p + "cls_token")
        self.mask_token = fp.view32(p + "mask_token") if (p + "mask_token") in fp.segments else None
        self.pos = fp.view32(p + "pos_embed") if self.abs_pos else None
        self.fcw, self.fcb = fp.view32(p + "fc_norm.weight"), fp.view32(p + "fc_norm.bias")

    def _g(self, i):
        gm, fp = self.gmap[i], self.fp
        return lambda k: fp.grad(gm[k])

    def forward(self, image, mask_u8=None, train=False, save=True, pre_mul=None, pool=True, twin=False):
        """image f32 [B,3,R,R] -> (y32 [B,N,D] f32, y16 bf16 same shape, state).  pool=False (tokenizer) leaves
        token 0 un-pooled.
        twin=True: the clean images AND their masked copies (mask_u8) run as ONE pass of 2B samples — rows [0, B) clean,
        [B, 2B) masked; the patch embedding is computed once.  Every GEMM / attention / LayerNorm launch of the encoder then
        serves both copies (the pre-training step encodes every image both ways, model_pretrain.py:43,73)."""
        if self.w is None:
            self.refresh()
        B0 = image.shape[0]
        N, D, npatch = self.N, self.D, self.np
        image = image.contiguous()
        cols = L.im2col(_f32(image), self.P, pre_mul)
        patch = L.gemm(cols, self.pe_w16, bias=self.pe_b, out_dtype=torch.float32)
        if twin:
            assert mask_u8 is not None
            B = 2 * B0
            x = torch.empty((B * N, D), dtype=torch.float32, device=patch.device)
            L.assemble_tokens(patch, self.cls, self.mask_token, None, self.pos, B0, npatch, out=x[:B0 * N])
            L.assemble_tokens(patch, self.cls, self.mask_token, mask_u8, self.pos, B0, npatch, out=x[B0 * N:])
        else:
            B = B0
            x = L.assemble_tokens(patch, self.cls, self.mask_token, mask_u8, self.pos, B, npatch)
        st = State()
        st.blocks = []
        ds_all = None
        if train and max(self.drop_path) > 0:
            # DropPath (beit2.py:35-45, one Bernoulli(keep) per sample per residual branch): all 2 x depth draws of the pass in
            # three launches instead of three per branch
            if getattr(self, "_keep", None) is None or self._keep.device != x.device:
                self._keep = torch.tensor([1.0 - p for p in self.drop_path], device=x.device).view(-1, 1, 1)
            ds_all = (torch.rand(self.depth, 2, B, device=x.device) < self._keep).float() / self._keep
        for i in range(self.depth):
            w = self.w[i]
            rb = L.relpos_bias_fwd(w["rel_table"], self.rel_index, N, self.H, self.bias_ld) if self.relbias else None
            ds = None
            if ds_all is not None and self.drop_path[i] > 0:
                ds = (ds_all[i, 0], ds_all[i, 1])
            rel = (w["rel_table"], self.ws) if (self.relbias and self.rel_closed_form) else None
            x, s = BK.vit_block_fwd(x, w, B, N, self.H, self.eps, relbias=rb, drop_scale=ds, save=save, rel=rel)
            st.blocks.append(s)
            if self.collect is not None:
                self.collect.append(x.view(B, N, D).clone())
        y16, stats, y32 = L.layernorm_fwd(x, self.fcw, self.fcb, self.eps, want_f32_copy=True, want_stats=save)
        if pool:
            L.meanpool_fwd_(y16, y32, B, npatch)
        if save:
            st.cols, st.mask, st.x_final, st.stats, st.B, st.twin = cols, mask_u8, x, stats, B, twin
        return y32.view(B, N, D), y16.view(B, N, D), (st if save else None)

    def backward(self, st, dy32, block_done=None):
        """dy32: f32 [B,N,D] gradient of the pooled output.  Accumulates every parameter gradient of the encoder.
        block_done(i), when given, is called as soon as block i's parameter gradients are final (kernels issued)."""
        B, N, D, npatch, p, fp = st.B, self.N, self.D, self.np, self.prefix, self.fp
        dy = L.meanpool_bwd(_f32(dy32).reshape(B * N, D).contiguous(), B, npatch)
        dx = L.layernorm_bwd(dy, st.x_final, st.stats, self.fcw, fp.grad(p + "fc_norm.weight"), fp.grad(p + "fc_norm.bias"))
        for i in reversed(range(self.depth)):
            dx = BK.vit_block_bwd(dx, st.blocks[i], self.w[i], self._g(i), B, N, self.H, rel_index=self.rel_index)
            st.blocks[i] = None  # free activations as we go
            if block_done is not None:
                block_done(i)
        dmask = fp.grad(p + "mask_token") if st.mask is not None else None
        if getattr(st, "twin", False):   # both copies read the same patch embedding: two accumulating wgrads, like two passes
            B0 = B // 2
            halves = ((dx[:B0 * N], None, None), (dx[B0 * N:], st.mask, dmask))
        else:
            B0 = B
            halves = ((dx, st.mask, dmask),)
        for dxh, mask, dm in halves:
            dpatch = L.assemble_tokens_bwd(dxh, mask, fp.grad(p + "cls_token"), dm, B0, npatch)
            L.colsum_into(dpatch, fp.grad(p + "patch_embed.proj.bias"))
            BK.wgrad(fp.grad(p + "patch_embed.proj.weight").view(D, -1), dpatch, st.cols)


# =====================================================================================================
# RoBERTa stack (text encoder / fusion encoder)
# =====================================================================================================
class RobertaStack:
    def __init__(self, fp, cfg, prefix, layers, cross, arch="roberta"):
        self.fp, self.cfg, self.prefix, self.layers, self.cross = fp, cfg, prefix, layers, cross
        self.names = TextNames(arch)
        self.D, self.H, self.eps, self.pad = cfg["hidden"], cfg["heads"], cfg["ln_eps"], cfg["pad_id"]
        self.w = None
        self.collect = None  # tests: list receiving a f32 copy of every layer output

    def refresh(self):
        fp, D = self.fp, self.D
        self.w, self.gmap = [], []
        for i in range(self.layers):
            l = f"{self.prefix}{self.names.stem}encoder.layer.{i}."
            a, c = l + "attention.", l + "crossattention."
            w = dict(qkv_w16=fp.span16(a + "self.query.weight", a + "self.value.weight", (3 * D, D)),
                     qkv_b=fp.span32(a + "self.query.bias", a + "self.value.bias", (3 * D,)),
                     a_o_w16=fp.view16(a + "output.dense.weight"), a_o_b=fp.view32(a + "output.dense.bias"),
                     a_ln_w=fp.view32(a + "output.LayerNorm.weight"), a_ln_b=fp.view32(a + "output.LayerNorm.bias"),
                     i_w16=fp.view16(l + "intermediate.dense.weight"), i_b=fp.view32(l + "intermediate.dense.bias"),
                     f_w16=fp.view16(l + "output.dense.weight"), f_b=fp.view32(l + "output.dense.bias"),
                     f_ln_w=fp.view32(l + "output.LayerNorm.weight"), f_ln_b=fp.view32(l + "output.LayerNorm.bias"))
            gm = dict(qkv_w=[a + f"self.{n}.weight" for n in ("query", "key", "value")],
                      qkv_b=[a + f"self.{n}.bias" for n in ("query", "key", "value")],
                      a_o_w=a + "output.dense.weight", a_o_b=a + "output.dense.bias", a_ln_w=a + "output.LayerNorm.weight",
                      a_ln_b=a + "output.LayerNorm.bias", i_w=l + "intermediate.dense.weight",
                      i_b=l + "intermediate.dense.bias", f_w=l + "output.dense.weight", f_b=l + "output.dense.bias",
                      f_ln_w=l + "output.LayerNorm.weight", f_ln_b=l + "output.LayerNorm.bias")
            if self.cross:
                Dk = fp.segments[c + "self.key.weight"].shape[1]
                w.update(c_q_w16=fp.view16(c + "self.query.weight"), c_q_b=fp.view32(c + "self.query.bias"),
                         c_kv_w16=fp.span16(c + "self.key.weight", c + "self.value.weight", (2 * D, Dk)),
                         c_kv_b=fp.span32(c + "self.key.bias", c + "self.value.bias", (2 * D,)),
                         c_o_w16=fp.view16(c + "output.dense.weight"), c_o_b=fp.view32(c + "output.dense.bias"),
                         c_ln_w=fp.view32(c + "output.LayerNorm.weight"), c_ln_b=fp.view32(c + "output.LayerNorm.bias"))
                gm.update(c_q_w=c + "self.query.weight", c_q_b=c + "self.query.bias",
                          c_kv_w=[c + "self.key.weight", c + "self.value.weight"],
                          c_kv_b=[c + "self.key.bias", c + "self.value.bias"], c_o_w=c + "output.dense.weight",
                          c_o_b=c + "output.dense.bias", c_ln_w=c + "output.LayerNorm.weight",
                          c_ln_b=c + "output.LayerNorm.bias")
            self.w.append(w)
            self.gmap.append(gm)
        e = self.prefix + self.names.stem + "embeddings."
        self.e = e
        self.word, self.posw, self.typew = (fp.view32(e + "word_embeddings.weight"), fp.view32(e + "position_embeddings.weight"),
                                            fp.view32(e + "token_type_embeddings.weight"))
        self.eln_w, self.eln_b = fp.view32(e + "LayerNorm.weight"), fp.view32(e + "LayerNorm.bias")

    def _g(self, i):
        gm, fp = self.gmap[i], self.fp

        def g(k):
            n = gm[k]
            if isinstance(n, list):
                seg = fp.segments[n[0]]
                shape = (len(n) * seg.shape[0],) + tuple(seg.shape[1:])
                return fp.span_grad(n, shape)
            return fp.grad(n)
        return g

    @staticmethod
    def additive_mask(atts):
        """xroberta.py:805-806: (1 - m) * -10000, f32 [B, L]."""
        return ((1.0 - atts.to(torch.float32)) * -10000.0).contiguous()

    def embed(self, ids, drop, save=True):
        if self.w is None:
            self.refresh()
        y, pre, stats, pos_ids = L.roberta_embed_fwd(ids.contiguous(), self.word, self.posw, self.typew, self.eln_w,
                                                     self.eln_b, self.pad, self.eps, want_pre=True,
                                                     absolute_pos=self.names.arch == "bert")
        st = State()
        st.ids, st.pre, st.stats, st.pos_ids, st.seed, st.p = ids, pre, stats, pos_ids, 0, drop.p_hidden
        y32 = None
        if drop.p_hidden > 0:  # xroberta.py:136
            st.seed = drop.next_seed()
            y = L.dropout_apply(y, drop.p_hidden, st.seed)
        elif pre is not None:  # f32 copy of the embedding output = residual of layer 0
            _, _, y32 = L.layernorm_fwd(pre, self.eln_w, self.eln_b, self.eps, want_f32_copy=True, want_stats=False)
        return y, y32, st

    def embed_bwd(self, st, dh):
        fp, e = self.fp, self.e
        if st.p > 0:
            dh = L.dropout_apply(dh.contiguous(), st.p, st.seed)
        dpre = L.layernorm_bwd(dh.contiguous(), st.pre, st.stats, self.eln_w, fp.grad(e + "LayerNorm.weight"),
                               fp.grad(e + "LayerNorm.bias"))
        L.roberta_embed_bwd(dpre, st.ids.reshape(-1), st.pos_ids, fp.grad(e + "word_embeddings.weight"),
                            fp.grad(e + "position_embeddings.weight"), fp.grad(e + "token_type_embeddings.weight"), self.pad,
                            pos_pad=-1 if self.names.arch == "bert" else self.pad)   # xbert.py:172-174 vs xroberta.py:92-102

    def layers_fwd(self, h, Bt, Lt, kmask, enc=None, Benc=0, Lenc=0, kv_index=None, drop=BK.NO_DROP, save=True, h32=None,
                   self_bias=None, enc_kmask=None, varlen=None):
        """Returns (h bf16 [Bt*Lt, D], h f32 same shape, state).  self_bias / enc_kmask: see blocks.roberta_layer_fwd.
        varlen: a Varlen batch packed into h's rows (Bt = 1, Lt = T, no kmask, no cross-attention)."""
        if self.w is None:
            self.refresh()
        assert varlen is None or (enc is None and kmask is None and self_bias is None and Bt == 1 and Lt == varlen.T)
        st = State()
        st.varlen = varlen
        st.layers, st.Bt, st.Lt, st.kmask, st.Benc, st.Lenc, st.kv_index = [], Bt, Lt, kmask, Benc, Lenc, kv_index
        st.kv_offsets = st.kv_samples = None
        st.self_bias, st.enc_kmask = self_bias, enc_kmask
        if enc is not None:  # CSR inverse of the sample -> image map: the tcgen05 cross-attention kernels stack an image's samples
            if kv_index is None:
                st.kv_offsets = torch.arange(Benc + 1, dtype=torch.int32, device=h.device)
                st.kv_samples = torch.arange(Bt, dtype=torch.int32, device=h.device)
            else:
                st.kv_offsets, st.kv_samples = csr_inverse(kv_index, Benc)
        # The cross-attention K | V projections of all layers read the same `enc`: one GEMM with the layers' weights stacked
        # along N (and, in the backward, one GEMM with them stacked along K for the gradient wrt `enc`: no fp32 read-modify-
        # write of the accumulator per layer) instead of one launch per layer.
        st.kvc_all = st.kv_wall = None
        kv_w = [w.get("c_kv_w16") for w in self.w]
        merged = enc is not None and self.layers > 1 and all(x is not None for x in kv_w) and MERGE_CROSS_KV
        D2 = 0
        if merged:
            D2 = kv_w[0].shape[0]
            st.kv_wall = torch.cat(kv_w, 0)
            st.kvc_all = L.gemm(enc, st.kv_wall, bias=torch.cat([w["c_kv_b"] for w in self.w]))
        for i in range(self.layers):
            h, h32, s = BK.roberta_layer_fwd(h, self.w[i], Bt, Lt, self.H, self.eps, kmask, enc=enc, Benc=Benc, Lenc=Lenc,
                                             kv_index=kv_index, drop=drop, save=save, h32=h32, kv_offsets=st.kv_offsets,
                                             kv_samples=st.kv_samples, self_bias=self_bias, enc_kmask=enc_kmask,
                                             kvc=st.kvc_all[:, i * D2:(i + 1) * D2] if merged else None, varlen=varlen)
            st.layers.append(s)
            if self.collect is not None:
                self.collect.append(h32.view(Bt, Lt, -1).clone())
        return h, h32, (st if save else None)

    @staticmethod
    def slice_states(est, st, B):
        """States of the first B samples of a pass that ran B' > B samples (no cross-attention): every saved tensor is
        per-row / per-sample and dropout masks are functions of (seed, sample, position), so the backward over the slice is
        the backward the B samples would have had on their own."""
        Bt, Lt = st.Bt, st.Lt

        def cut(v):
            if torch.is_tensor(v) and v.dim() >= 1:
                if v.shape[0] == Bt * Lt:
                    return v[:B * Lt]
                if v.shape[0] == Bt:
                    return v[:B]
            return v
        out = State()
        out.__dict__.update({k: cut(v) for k, v in st.__dict__.items()})
        out.Bt = B
        out.layers = []
        for s in st.layers:
            c = BK.Saved()
            c.__dict__.update({k: cut(v) for k, v in s.__dict__.items()})
            out.layers.append(c)
        e = State()
        e.__dict__.update({k: cut(v) for k, v in est.__dict__.items()})
        return e, out

    def layers_bwd(self, st, dh, d_enc=None, need_dh=True, kv_offsets=None, kv_samples=None, d_enc_fresh=False):
        """dh: bf16 / f32 [Bt*Lt, D].  d_enc: f32 [Benc*Lenc, Denc] accumulator (cross-attention K/V input gradient);
        d_enc_fresh: it is uninitialised memory that the merged K | V gradient GEMM may simply overwrite."""
        if kv_samples is None:   # CSR built in layers_fwd (identity when every sample has its own image)
            kv_offsets, kv_samples = st.kv_offsets, st.kv_samples
        kvc_all = getattr(st, "kvc_all", None)
        dkvc_all = torch.empty_like(kvc_all) if kvc_all is not None else None
        D2 = kvc_all.shape[1] // self.layers if kvc_all is not None else 0
        for i in reversed(range(self.layers)):
            last = i == 0
            dh = BK.roberta_layer_bwd(dh, st.layers[i], self.w[i], self._g(i), st.Bt, st.Lt, self.H, st.kmask, Benc=st.Benc,
                                      Lenc=st.Lenc, kv_index=st.kv_index, kv_offsets=kv_offsets, kv_samples=kv_samples,
                                      d_enc=d_enc, need_dh=(need_dh or not last), self_bias=st.self_bias,
                                      enc_kmask=st.enc_kmask,
                                      dkvc_out=dkvc_all[:, i * D2:(i + 1) * D2] if dkvc_all is not None else None,
                                      varlen=getattr(st, "varlen", None))
            st.layers[i] = None
        if dkvc_all is not None and d_enc is not None:   # gradient wrt the image tokens: all layers in one long-K GEMM
            L.gemm(dkvc_all, st.kv_wall, b_t=True, out=d_enc, accumulate=not d_enc_fresh)
        st.kvc_all = st.kv_wall = None
        return dh


class Varlen:
    """A packed variable-length batch: n sequences of 1..128 tokens back to back in T rows.  cu / tiles: int32 device copies
    of lib.varlen_plan (row offsets, tiles of the packed attention kernels); Lpad: the padded length the batch arrived in,
    which numbers the attention dropout mask as in the padded layout."""

    def __init__(self, lengths, Lpad, device):
        cu, tiles = L.varlen_plan(lengths)
        self.n, self.T, self.Lpad = cu.numel() - 1, int(cu[-1]), int(Lpad)
        self.cu, self.tiles = cu.to(device, non_blocking=True), tiles.to(device, non_blocking=True)


MERGE_CROSS_KV = __import__("os").environ.get("XFM_MERGE_CROSS_KV", "1") != "0"   # A/B switch for measurements


def csr_inverse(kv_index, Bkv):
    """CSR inverse of a sample -> K/V row map (int32 device tensors): rows of kv_samples grouped by K/V row."""
    order = torch.argsort(kv_index.long(), stable=True).to(torch.int32)
    counts = torch.zeros(Bkv, dtype=torch.int64, device=kv_index.device)  # bincount would sync to size its output
    counts.scatter_add_(0, kv_index.long(), torch.ones_like(kv_index, dtype=torch.int64))
    offsets = torch.zeros(Bkv + 1, dtype=torch.int32, device=kv_index.device)
    offsets[1:] = torch.cumsum(counts, 0).to(torch.int32)
    return offsets, order


# =====================================================================================================
# heads
# =====================================================================================================
def cls_rows(h16, B, Lt):
    """[B*Lt, D] -> strided [B, D] view of token 0 of every sample (a valid TMA operand: row stride Lt*D)."""
    D = h16.shape[-1]
    return h16.reshape(B, Lt * D)[:, :D]


class ProjHead:
    """F.normalize(Linear(x[:, 0, :])) (xfm.py:614-621), in exact fp32: the op is latency-bound ([B,768]x[768,E]) and its
    rounding error is multiplied by 1/temp (~14x) in the contrastive logits."""

    def __init__(self, fp, name):
        self.fp, self.name = fp, name

    def forward(self, emb32, B, Lt):
        fp, n = self.fp, self.name
        D = emb32.shape[-1]
        x0 = emb32.reshape(B, Lt * D)[:, :D]
        z = L.sgemm_f32(x0, fp.view32(n + ".weight"), bias=fp.view32(n + ".bias"))
        y, inv = L.l2norm_fwd(z)
        st = State()
        st.x0, st.y, st.inv, st.B, st.Lt = x0, y, inv, B, Lt
        return y, st

    def backward(self, st, dy):
        """Returns d_emb f32 [B, Lt, D] (non-zero only at token 0)."""
        fp, n = self.fp, self.name
        dz = L.l2norm_bwd(_f32(dy).contiguous(), st.y, st.inv)
        ones = torch.ones((1, st.B), dtype=torch.float32, device=dz.device)
        L.sgemm_f32(dz.t(), ones, out=fp.grad(n + ".bias").view(-1, 1), accumulate=True)  # db[E] += sum_b dz[b,:]
        L.sgemm_f32(dz.t(), st.x0.t(), out=fp.grad(n + ".weight"), accumulate=True)   # dW[E,D] += dz^T x0
        D = st.x0.shape[1]
        d_emb = torch.zeros((st.B, st.Lt * D), dtype=torch.float32, device=dz.device)
        L.sgemm_f32(dz, fp.view32(n + ".weight").t(), out=d_emb[:, :D])              # dx0[B,D] = dz W
        return d_emb.view(st.B, st.Lt, D)


class MlpHead:
    """build_mlp (xfm.py:115-121) followed by cross-entropy: itm_head on the fusion CLS rows (xfm.py:795-802)."""

    def __init__(self, fp, name, nout):
        self.fp, self.name, self.nout = fp, name, nout

    def logits(self, x0, save=True):
        fp, n = self.fp, self.name
        z = L.gemm(x0, fp.view16(n + ".0.weight"), bias=fp.view32(n + ".0.bias"), out_dtype=torch.float32)
        zn, stats, _ = L.layernorm_fwd(z, fp.view32(n + ".1.weight"), fp.view32(n + ".1.bias"), 1e-5, out_dtype=torch.float32,
                                       want_stats=save)
        a = L.gelu_fwd(zn)
        logits = L.gemm(a, fp.view16(n + ".3.weight"), bias=fp.view32(n + ".3.bias"), out_dtype=torch.float32)
        st = State()
        st.x0, st.z, st.zn, st.stats, st.a, st.logits = x0, z, zn, stats, a, logits
        return logits, st

    def backward(self, st, dlogits16, dx_out):
        """dlogits16: bf16 [R, 8] (zero padded beyond nout).  Writes the gradient wrt x0 into dx_out (bf16 strided view)."""
        fp, n, no = self.fp, self.name, self.nout
        L.colsum_into(dlogits16, fp.grad_padded(n + ".3.bias", 8))
        BK.wgrad(fp.grad(n + ".3.weight"), dlogits16[:, :no], st.a)
        da = L.gemm(dlogits16[:, :no], fp.view16(n + ".3.weight"), b_t=True)
        dzn = L.gelu_bwd(da, st.zn)
        dz = L.layernorm_bwd(dzn, st.z, st.stats, fp.view32(n + ".1.weight"), fp.grad(n + ".1.weight"), fp.grad(n + ".1.bias"),
                             out_dtype=torch.bfloat16)
        L.colsum_into(dz, fp.grad(n + ".0.bias"))
        BK.wgrad(fp.grad(n + ".0.weight"), dz, st.x0)
        L.gemm(dz, fp.view16(n + ".0.weight"), b_t=True, out=dx_out)


class LMHead:
    """RobertaLMHead (xroberta.py:1313-1333) with the decoder tied to the word embeddings, fused with
    CE(ignore_index=-100) (xroberta.py:1298-1299).  The f32 logits are materialised once ([R, V] padded to 8)."""

    def __init__(self, fp, cfg, prefix, arch="roberta", head="lm_head"):
        self.fp, self.cfg, self.p = fp, cfg, prefix
        self.V, self.eps = cfg["vocab_size"], cfg["ln_eps"]
        self.ldv = (self.V + 7) // 8 * 8
        names = TextNames(arch)
        self.n = {k: prefix + v for k, v in names.head(head).items()}
        self.word = prefix + names.stem + "embeddings.word_embeddings.weight"

    def logits(self, x, st=None):
        """x bf16 [R, D] -> f32 logits [R, ldv] (columns >= V are padding)."""
        fp, p = self.fp, self.p
        R = x.shape[0]
        pre = torch.empty_like(x)
        n = self.n
        a = L.gemm(x, fp.view16(n["dense_w"]), bias=fp.view32(n["dense_b"]), act=1, aux_out=pre)
        y, stats, _ = L.layernorm_fwd(a, fp.view32(n["ln_w"]), fp.view32(n["ln_b"]), self.eps)
        logits = torch.empty((R, self.ldv), dtype=torch.float32, device=x.device)
        L.gemm(y, fp.view16(self.word), bias=fp.view32(n["bias"]), out=logits[:, :self.V])
        if st is not None:
            st.x, st.pre, st.a, st.y, st.stats, st.logits = x, pre, a, y, stats, logits
        return logits

    def loss(self, x, labels):
        """x bf16 [R, D] gathered hidden rows; labels int64 [R]."""
        st = State()
        logits = self.logits(x, st)
        loss, count, lse = L.ce_fwd(logits, labels, self.V)
        st.labels, st.count, st.lse = labels, count, lse
        return loss, st

    def loss_rows(self, x, labels):
        """CrossEntropyLoss(reduction='none') (xroberta.py:1108-1109): per-row losses f32 [R] (0 where label = -100)."""
        st = State()
        logits = self.logits(x, st)
        _, count, lse, rows = L.ce_fwd(logits, labels, self.V, want_rows=True)
        st.labels, st.count, st.lse = labels, count, lse
        return rows, st

    def backward(self, st, upstream, row_scale=None):
        """upstream: f32 [1] device scalar (or None = 1); row_scale: f32 [R] gradient of the scalar loss wrt each row loss
        (loss_rows), else the mean reduction of loss().  Returns d_x bf16 [R, D]."""
        fp, p, V = self.fp, self.p, self.V
        if row_scale is not None:
            dlog = L.ce_bwd_rows(st.logits, st.labels, st.lse, row_scale, upstream, V, self.ldv)
        else:
            dlog = L.ce_bwd(st.logits, st.labels, st.lse, st.count, upstream, V, self.ldv)
        st.logits = None
        n = self.n
        L.colsum_into(dlog, fp.grad_padded(n["bias"], self.ldv))
        BK.wgrad(fp.grad(self.word), dlog[:, :V], st.y)
        dy = L.gemm(dlog[:, :V], fp.view16(self.word), b_t=True)
        da = L.layernorm_bwd(dy, st.a, st.stats, fp.view32(n["ln_w"]), fp.grad(n["ln_w"]), fp.grad(n["ln_b"]),
                             out_dtype=torch.bfloat16)
        dpre = L.gelu_bwd(da, st.pre)
        L.colsum_into(dpre, fp.grad(n["dense_b"]))
        BK.wgrad(fp.grad(n["dense_w"]), dpre, st.x)
        return L.gemm(dpre, fp.view16(n["dense_w"]), b_t=True)


class LinearCE:
    """nn.Linear + CrossEntropyLoss on gathered rows: the VQ-KD MIM head (xfm.py:494-496,629)."""

    def __init__(self, fp, name, nout):
        self.fp, self.name, self.nout = fp, name, nout

    def loss(self, x, labels):
        fp, n = self.fp, self.name
        logits = L.gemm(x, fp.view16(n + ".weight"), bias=fp.view32(n + ".bias"), out_dtype=torch.float32)
        loss, count, lse = L.ce_fwd(logits, labels, self.nout)
        st = State()
        st.x, st.logits, st.labels, st.count, st.lse = x, logits, labels, count, lse
        return loss, st

    def backward(self, st, upstream):
        fp, n = self.fp, self.name
        dlog = L.ce_bwd(st.logits, st.labels, st.lse, st.count, upstream, self.nout, self.nout)
        L.colsum_into(dlog, fp.grad(n + ".bias"))
        BK.wgrad(fp.grad(n + ".weight"), dlog, st.x)
        return L.gemm(dlog, fp.view16(n + ".weight"), b_t=True)
