"""RoBERTa sequence classification (transformers' RobertaForSequenceClassification, what the reference's run_glue.py
fine-tunes) on the C-ABI kernels: a drop-in for GLUE fine-tuning of the X-FM text encoder.

    model = RobertaForSequenceClassification.from_pretrained(model_dir, num_labels=3).to("cuda")

Parameters live in one flat fp32 buffer with a bf16 shadow (params.FlatParams); state_dict() names and shapes are
transformers'.  The parameters are views of that buffer, so a torch.optim.AdamW built over model.parameters() (what HF's
Trainer builds) updates it in place, and the next forward recasts the shadow because the parameters' version counters
moved.
FlatAdamW(model) works too.

Batches arrive padded to max_seq_length while most GLUE sentences are much shorter.  When every sequence keeps at most 128
tokens, the forward packs the kept tokens (attention_mask == 1) of all sequences back to back: the GEMMs, LayerNorms and
dropouts of the encoder run on real tokens only and the self-attention runs on the packed variable-length tcgen05 kernels
(csrc/attention_vtc.cu).  Masked tokens are never keys and only token 0 is classified, so packing gives HF's result for
masks with holes too.  Reading the lengths costs one device -> host copy per forward (the packed size T and the tile table
depend on them), so this path is not CUDA-graph capturable.  A batch with a longer sequence runs the padded encoder with
its additive key mask.
"""
import json
import os
import types
from collections import OrderedDict

import torch
from torch import nn

from . import blocks as BK
from . import checkpoint as CK
from . import encoders as E
from . import lib as L
from .params import FlatParams
from .xfm import _Holder

VARLEN_MAX = 128   # longest sequence the packed attention kernels take (xfm_attention_varlen_plan)

_CONFIG_KEYS = dict(vocab_size=50265, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                    hidden_act="gelu", hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, max_position_embeddings=514,
                    type_vocab_size=1, initializer_range=0.02, layer_norm_eps=1e-5, pad_token_id=1, classifier_dropout=None,
                    num_labels=2, problem_type=None)


def _config(config, overrides=None):
    """RobertaConfig (or its dict) -> SimpleNamespace with the attributes this model reads."""
    d = config.to_dict() if hasattr(config, "to_dict") else dict(config or {})
    d.update(overrides or {})
    if "num_labels" not in d and "id2label" in d:
        d["num_labels"] = len(d["id2label"])
    c = types.SimpleNamespace(**{k: d.get(k, v) for k, v in _CONFIG_KEYS.items()})
    if c.hidden_size != 64 * c.num_attention_heads:
        raise ValueError("head_dim must be 64 (hidden_size = 64 * num_attention_heads)")
    if c.hidden_act != "gelu":
        raise ValueError("hidden_act must be 'gelu' (erf form)")
    return c


class SequenceClassifierOutput(OrderedDict):
    """What HF's Trainer reads: .loss / .logits, ["loss"], and index 0 = loss when labels were given (else logits)."""

    def __init__(self, loss=None, logits=None):
        super().__init__()
        if loss is not None:
            self["loss"] = loss
        self["logits"] = logits

    def __getattr__(self, k):
        if k in ("loss", "logits"):
            return self.get(k)
        raise AttributeError(k)

    def __getitem__(self, k):
        if isinstance(k, (int, slice)):
            return tuple(self.values())[k]
        return super().__getitem__(k)

    def to_tuple(self):
        return tuple(self.values())


class _ClassifyFn(torch.autograd.Function):
    """One autograd node per forward: (loss, logits) from the anchor; backward accumulates every parameter gradient into
    the flat gradient buffer."""

    @staticmethod
    def forward(ctx, impl, anchor):
        ctx.set_materialize_grads(False)
        ctx.impl = impl
        return impl.fwd()

    @staticmethod
    def backward(ctx, g_loss, g_logits):
        ctx.impl.bwd(g_loss, g_logits)
        return None, None


class RobertaForSequenceClassification(nn.Module):
    def __init__(self, config, init_seed=0, device="cpu"):
        super().__init__()
        c = self.config = _config(config)
        if c.problem_type not in (None, "regression", "single_label_classification", "multi_label_classification"):
            raise ValueError("unknown problem_type %r" % (c.problem_type,))
        self.num_labels = c.num_labels
        D = c.hidden_size
        self._cfg = dict(hidden=D, ffn=c.intermediate_size, vocab_size=c.vocab_size, max_pos=c.max_position_embeddings,
                         type_vocab=c.type_vocab_size, heads=c.num_attention_heads, ln_eps=c.layer_norm_eps,
                         pad_id=c.pad_token_id)
        fp = self.flat = FlatParams()
        E.add_roberta(fp, self._cfg, self._hf_init(init_seed), "", c.num_hidden_layers, cross=False, enc_width=D, heads=())
        init = self._hf_init(init_seed + 1)
        for n, shape in (("classifier.dense.weight", (D, D)), ("classifier.dense.bias", (D,)),
                         ("classifier.out_proj.weight", (c.num_labels, D)), ("classifier.out_proj.bias", (c.num_labels,))):
            fp.add(n, shape, init=init(n, shape))
        fp.finalize(torch.device(device))
        self._params = OrderedDict()
        for name in fp.segments:
            p = nn.Parameter(fp.view32(name))
            self._params[name] = p
            *path, leaf = name.split(".")
            mod = self
            for part in path:
                if part not in mod._modules:
                    mod.add_module(part, _Holder())
                mod = mod._modules[part]
            mod.register_parameter(leaf, p)
        self._enc = E.RobertaStack(fp, self._cfg, "", c.num_hidden_layers, cross=False)
        self._anchor = torch.zeros((), requires_grad=True)
        self._seed = int(torch.initial_seed()) & 0x7FFFFFFF
        self._calls = 0
        self._param_version = None

    # ------------------------------------------------------------------ parameters
    def _hf_init(self, seed):
        """RobertaPreTrainedModel._init_weights: normal(0, initializer_range) weights and embeddings (padding row zero),
        zero biases, unit LayerNorm."""
        g = torch.Generator().manual_seed(seed)
        std, pad = self.config.initializer_range, self.config.pad_token_id

        def init(name, shape):
            if "LayerNorm" in name:
                return torch.ones(shape) if name.endswith("weight") else torch.zeros(shape)
            if name.endswith("bias"):
                return torch.zeros(shape)
            w = torch.empty(shape).normal_(0.0, std, generator=g)
            if name.endswith(("word_embeddings.weight", "position_embeddings.weight")) and 0 <= pad < shape[0]:
                w[pad] = 0.0
            return w
        return init

    def flat_buffers(self):
        return [(self.flat, self._params)]

    def adopt_stray_parameters(self):
        stray = [n for n, p in self.named_parameters() if all(p is not q for q in self._params.values())]
        if stray:
            raise RuntimeError("parameters outside the flat buffer: " + ", ".join(stray[:4]))

    def collect_stray_grads(self):
        pass

    def zero_grad(self, set_to_none=True):
        self.flat.zero_grad()
        for p in self._params.values():
            p.grad = None

    def _apply(self, fn, recurse=True):
        """.to(device) / .cuda() move the flat buffer and re-point every parameter view; dtype changes are refused (fp32
        master weights, bf16 compute is internal)."""
        if self.flat.move(fn):
            with torch.no_grad():
                for name, p in self._params.items():
                    p.data = self.flat.view32(name)
                    p.grad = None
            self._enc.w = None
        return self

    def load_state_dict(self, state_dict, strict=True, assign=False):
        out = super().load_state_dict(state_dict, strict=strict, assign=False)
        self.flat.sync_shadow(force=True)
        return out

    def _init_missing_classifier(self, missing):
        """Classifier weights a checkpoint lacks start as HF starts them: normal(0, initializer_range), zero biases."""
        init = self._hf_init(int(torch.initial_seed()) & 0x7FFFFFFF)
        with torch.no_grad():
            for n in missing:
                if n.startswith("classifier."):
                    seg = self.flat.segments[n]
                    self.flat.view32(n).copy_(init(n, seg.shape))
        self.flat.sync_shadow(force=True)

    @classmethod
    def from_pretrained(cls, model_dir, device="cpu", **config_overrides):
        """<dir>/config.json + <dir>/pytorch_model.bin (a RobertaForMaskedLM or RobertaForSequenceClassification
        checkpoint); config_overrides (num_labels, problem_type, dropouts, ...) take precedence over config.json."""
        with open(os.path.join(model_dir, "config.json")) as f:
            cfg = json.load(f)
        cfg.update(config_overrides)
        model = cls(cfg, device=device)
        state = CK.text_init_state(model_dir, model.config.num_hidden_layers, "roberta")
        sd = {}
        for k, v in state.items():
            k = k[len("text_encoder."):]
            if k.startswith(("roberta.embeddings.", "roberta.encoder.")) or k.startswith("classifier."):
                if k in model.flat.segments and tuple(v.shape) == model.flat.segments[k].shape:
                    sd[k] = v
        msg = model.load_state_dict(sd, strict=False)
        model._init_missing_classifier(msg.missing_keys)
        return model

    @classmethod
    def from_xfm_checkpoint(cls, path, config, device="cpu"):
        """The text encoder of an X-FM checkpoint (pre-training spelling text_encoder.roberta.*, fine-tuning spelling
        text_encoder.embeddings.* / text_encoder.encoder.*) as roberta.*; a fresh classifier."""
        model = cls(config, device=device)
        ck = torch.load(path, map_location="cpu") if isinstance(path, (str, os.PathLike)) else path
        ck = ck.get("model", ck)
        msg = model.load_state_dict(xfm_text_state(ck), strict=False)
        model._init_missing_classifier(msg.missing_keys)
        return model

    # ------------------------------------------------------------------ forward
    def _drop(self):
        c = self.config
        if not self.training:
            return BK.NO_DROP, 0.0
        self._calls += 1
        pc = c.classifier_dropout if c.classifier_dropout is not None else c.hidden_dropout_prob
        return BK.DropCfg(c.hidden_dropout_prob, c.attention_probs_dropout_prob, self._seed * 131 + self._calls), float(pc)

    def forward(self, input_ids, attention_mask=None, token_type_ids=None, labels=None, **ignored):
        if self.flat.P.device.type != "cuda":
            raise RuntimeError("RobertaForSequenceClassification runs on the GPU: call .to('cuda') first")
        dev = self.flat.P.device
        # An optimizer over model.parameters() (HF's Trainer builds torch.optim.AdamW) writes the parameters in place.  After
        # .to(device) they are views of the flat buffer with version counters of their own (p.data = ... keeps a tensor's
        # counter), so the bf16 shadow is recast when any parameter's counter moved, not only the buffer's.
        ver = sum(p._version for p in self._params.values())
        self.flat.sync_shadow(force=ver != self._param_version)
        self._param_version = ver
        ids = input_ids.to(dev, torch.int64).contiguous()
        B, Lp = ids.shape
        m = torch.ones_like(ids, dtype=torch.bool) if attention_mask is None else attention_mask.to(dev) != 0
        # the one device -> host read of the forward: kept tokens per row, whether token 0 is kept, token types
        info = [m.sum(1), m[:, 0].long()]
        if token_type_ids is not None:
            info.append((token_type_ids.to(dev) != 0).any().long().view(1))
        info = torch.cat(info).cpu()
        lengths, first = info[:B], info[B:2 * B]
        if token_type_ids is not None and int(info[2 * B]):
            raise ValueError("token_type_ids must be all zero: RoBERTa has one token type")
        if int(lengths.min()) == 0:
            raise ValueError("attention_mask has an all-zero row")
        if int(first.min()) == 0:
            raise ValueError("attention_mask masks token 0 of a row (token 0 is the one classified)")
        problem = self._problem(labels)
        impl = _Impl(self, ids, m, lengths, labels, problem, save=torch.is_grad_enabled())
        loss, logits = _ClassifyFn.apply(impl, self._anchor) if impl.save else impl.fwd()
        return SequenceClassifierOutput(loss=loss if labels is not None else None, logits=logits)

    def _problem(self, labels):
        """HF's problem_type rule."""
        c = self.config
        if labels is None:
            return None
        pt = c.problem_type
        if pt is None:
            if self.num_labels == 1:
                pt = "regression"
            elif labels.dtype in (torch.long, torch.int):
                pt = "single_label_classification"
            else:
                pt = "multi_label_classification"
        if pt == "multi_label_classification":
            raise NotImplementedError("multi-label classification is not supported (GLUE does not use it)")
        return pt


class _Impl:
    def __init__(self, model, ids, m, lengths, labels, problem, save):
        self.model, self.ids, self.m, self.lengths, self.labels, self.problem = model, ids, m, lengths, labels, problem
        self.save = save   # grad mode of the caller (autograd.Function.forward runs with grad mode off)

    def fwd(self):
        model, ids, m = self.model, self.ids, self.m
        stack, fp, c = model._enc, model.flat, model.config
        B, Lp = ids.shape
        dev = ids.device
        drop, pc = model._drop()
        save = self.save
        y, y32, est = stack.embed(ids, drop, save=save)
        if int(self.lengths.max()) <= VARLEN_MAX:
            # kept rows of the padded layout in order (a stable sort: no data-dependent output size, no second sync)
            rows = torch.argsort((~m).view(-1).to(torch.uint8), stable=True)[:int(self.lengths.sum())].contiguous()
            V = E.Varlen(self.lengths, Lp, dev)
            h = L.gather_rows(y, rows)
            h32 = L.gather_rows(y32, rows) if y32 is not None else None
            h, h32, st = stack.layers_fwd(h, 1, V.T, None, drop=drop, save=save, h32=h32, varlen=V)
            cls_rows = V.cu[:-1].long()
        else:
            rows = None
            kmask = E.RobertaStack.additive_mask(m)
            h, h32, st = stack.layers_fwd(y, B, Lp, kmask, drop=drop, save=save, h32=y32)
            cls_rows = torch.arange(B, device=dev) * Lp
        D = h.shape[1]
        nl = model.num_labels
        x0 = L.gather_rows(h, cls_rows)
        s1 = s2 = 0
        if pc > 0:
            s1, s2 = drop.next_seed(), drop.next_seed()
            x0 = L.dropout_apply(x0, pc, s1)
        a32 = L.gemm(x0, fp.view16("classifier.dense.weight"), bias=fp.view32("classifier.dense.bias"), act=3,
                     out_dtype=torch.float32)
        a = torch.empty(a32.shape, dtype=torch.bfloat16, device=dev)
        L.cast_to_bf16(a32, a)
        if pc > 0:
            a = L.dropout_apply(a, pc, s2)
        ld = (nl + 7) // 8 * 8
        logits_pad = torch.empty((B, ld), dtype=torch.float32, device=dev)
        L.gemm(a, fp.view16("classifier.out_proj.weight"), bias=fp.view32("classifier.out_proj.bias"), out=logits_pad[:, :nl])
        logits = logits_pad[:, :nl]
        loss = torch.zeros((), dtype=torch.float32, device=dev)
        self.ce = None
        if self.problem == "regression":
            lab = self.labels.to(dev, torch.float32).reshape(B)
            self.diff = logits[:, 0] - lab if nl == 1 else None
            if nl != 1:
                raise ValueError("regression needs num_labels == 1")
            loss = (self.diff * self.diff).mean()
        elif self.problem == "single_label_classification":
            lab = self.labels.to(dev, torch.int64).reshape(B).contiguous()
            l1, count, lse = L.ce_fwd(logits_pad, lab, nl)
            self.ce = (lab, count, lse)
            loss = l1.view(())
        if save:
            self.st, self.est, self.rows, self.cls_rows, self.T = st, est, rows, cls_rows, h.shape[0]
            self.x0, self.a32, self.a, self.logits_pad, self.pc, self.s1, self.s2, self.ld = x0, a32, a, logits_pad, pc, s1, s2, ld
        return loss.detach().clone(), logits.detach().clone()

    def bwd(self, g_loss, g_logits):
        model = self.model
        fp, stack, nl, ld = model.flat, model._enc, model.num_labels, self.ld
        if any(p.grad is None or p.grad.data_ptr() != fp._view(fp.G, n).data_ptr()
               for n, p in model._params.items()):
            fp.zero_grad()   # first backward, or the optimizer dropped the gradients (zero_grad(set_to_none=True))
        dev = self.x0.device
        B = self.x0.shape[0]
        dl = torch.zeros((B, ld), dtype=torch.float32, device=dev)
        if g_logits is not None:
            dl[:, :nl] += g_logits
        if g_loss is not None and self.problem == "single_label_classification":
            lab, count, lse = self.ce
            dl += L.ce_bwd(self.logits_pad, lab, lse, count, g_loss.reshape(1).float().contiguous(), nl, ld).float()
        elif g_loss is not None and self.problem == "regression":
            dl[:, 0] += self.diff * (2.0 / B) * g_loss
        dlog = dl.to(torch.bfloat16)
        L.colsum_into(dlog, fp.grad_padded("classifier.out_proj.bias", ld))
        BK.wgrad(fp.grad("classifier.out_proj.weight"), dlog[:, :nl], self.a)
        da = L.gemm(dlog[:, :nl], fp.view16("classifier.out_proj.weight"), b_t=True)
        if self.pc > 0:
            da = L.dropout_apply(da, self.pc, self.s2)
        dz = (da.float() * (1.0 - self.a32 * self.a32)).to(torch.bfloat16)   # tanh' on the [B, D] classified rows
        L.colsum_into(dz, fp.grad("classifier.dense.bias"))
        BK.wgrad(fp.grad("classifier.dense.weight"), dz, self.x0)
        dx0 = L.gemm(dz, fp.view16("classifier.dense.weight"), b_t=True)
        if self.pc > 0:
            dx0 = L.dropout_apply(dx0, self.pc, self.s1)
        D = dx0.shape[1]
        dh = torch.zeros((self.T, D), dtype=torch.float32, device=dev)
        L.scatter_add_rows_(dh, self.cls_rows, dx0)
        dh = stack.layers_bwd(self.st, dh)
        if self.rows is not None:
            dy = torch.zeros((self.ids.numel(), D), dtype=torch.float32, device=dev)
            L.scatter_add_rows_(dy, self.rows, dh)
        else:
            dy = dh
        stack.embed_bwd(self.est, dy)
        with torch.no_grad():
            for n, p in model._params.items():
                if p.grad is None:
                    p.grad = fp._view(fp.G, n)
        self.st = self.est = None


def xfm_text_state(state):
    """X-FM checkpoint keys -> RobertaForSequenceClassification keys: text_encoder.roberta.<x> (pre-training) and
    text_encoder.<x> for x under embeddings. / encoder. (fine-tuning models hold a bare RobertaModel) become roberta.<x>;
    every other key is dropped."""
    out = {}
    for k, v in state.items():
        if k.startswith("text_encoder.roberta."):
            out["roberta." + k[len("text_encoder.roberta."):]] = v
        elif k.startswith(("text_encoder.embeddings.", "text_encoder.encoder.")):
            out["roberta." + k[len("text_encoder."):]] = v
    return out
