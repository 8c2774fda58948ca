"""Helper for tests/test_boundary_cpu.py — run as a SUBPROCESS (it rebinds `models` in sys.modules), only where
XFM_REFERENCE_ROOT names a checkout of the original XFM sources.  Prints one JSON object.

    python tests/ref_probe.py loaders    constructor-time checkpoint import: reference XFM(load_*_params=True) vs xfm_b200
    python tests/ref_probe.py subclass   the reference's OWN models/model_pretrain.py, model_retrieval.py and model_nlvr.py
                                         source, subclassing xfm_b200.XFMBase through sys.modules['models.xfm']
"""
import importlib.util
import json
import os
import sys
import tempfile
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.environ.get("XFM_REFERENCE_ROOT", "")

from oracle import ref_shim  # noqa: E402
from oracle import xfm_oracle as O  # noqa: E402


def synth_checkpoints(cfg, src_window=6):
    """A RoBERTa-for-MLM checkpoint directory (HF key layout) and a BEiT-v2 checkpoint saved at ANOTHER resolution with one
    shared relative-position table — the two files the reference's constructor reads."""
    g = torch.Generator().manual_seed(5)
    tdir = ref_shim.roberta_config_dir(cfg)
    text = {}
    for name, shape in O.param_shapes(cfg).items():
        if name.startswith("text_encoder.") and "lm_cap_head" not in name:
            text[name[len("text_encoder."):]] = torch.randn(shape, generator=g) * 0.05
    text["lm_head.decoder.weight"] = text["roberta.embeddings.word_embeddings.weight"]
    text["roberta.embeddings.position_ids"] = torch.arange(cfg["max_pos"]).expand((1, -1)).clone()
    text["roberta.pooler.dense.weight"] = torch.randn(cfg["hidden"], cfg["hidden"], generator=g)
    text["roberta.pooler.dense.bias"] = torch.randn(cfg["hidden"], generator=g)
    torch.save(text, os.path.join(tdir, "pytorch_model.bin"))
    vis = {}
    for name, shape in O.param_shapes(cfg).items():
        if name.startswith("vision_encoder.") and "relative_position" not in name:
            vis[name[len("vision_encoder."):]] = torch.randn(shape, generator=g) * 0.05
    H = cfg["vision_heads"]
    vis["rel_pos_bias.relative_position_bias_table"] = torch.randn((2 * src_window - 1) ** 2 + 3, H, generator=g)
    vis["blocks.0.attn.relative_position_index"] = torch.zeros(src_window ** 2 + 1, src_window ** 2 + 1, dtype=torch.long)
    vis["head.weight"] = torch.randn(10, cfg["vision_width"], generator=g)
    vis["head.bias"] = torch.randn(10, generator=g)
    f = tempfile.NamedTemporaryFile(suffix=".pth", delete=False)
    torch.save({"model": vis}, f.name)
    return tdir, f.name


def our_config(cfg, tdir, vckpt):
    vdir = tempfile.mkdtemp(prefix="beit2-base-")
    vpath = os.path.join(vdir, "config_beit2_base.json")
    with open(vpath, "w") as fh:
        json.dump(dict(ckpt=vckpt, vision_width=cfg["vision_width"], patch_size=cfg["patch_size"]), fh)
    c = dict(cfg)
    c.update(use_beit_v2=True, vision_config=vpath, text_encoder=tdir, text_num_hidden_layers=cfg["text_layers"],
             text_fusion_start_at=cfg["text_layers"], fusion_num_hidden_layers=cfg["fusion_layers"], fusion_fusion_start_at=0,
             local_attn_depth=-1, accelerator=dict(FP16_OPT_LEVEL="O1"))
    return c


def loaders():
    cfg = O.tiny_config()
    tdir, vckpt = synth_checkpoints(cfg)
    ref = ref_shim.build_reference_xfm(cfg, None, load_vision_params=True, load_text_params=True, vision_ckpt=vckpt, text_dir=tdir)
    from xfm_b200.model_pretrain import XFM
    torch.manual_seed(0)
    mine = XFM(our_config(cfg, tdir, vckpt), load_vision_params=True, load_text_params=True, device="cpu")
    rsd, msd = ref.state_dict(), mine.state_dict()
    loaded, worst, missing = 0, 0.0, []
    for k, v in rsd.items():
        if k not in msd:
            missing.append(k)
            continue
        if k.startswith(("vision_encoder.", "text_encoder.roberta.", "text_encoder.lm_head.")) and v.dtype.is_floating_point:
            loaded += 1
            worst = max(worst, float((v - msd[k]).abs().max()))
    tbl = "vision_encoder.blocks.1.attn.relative_position_bias_table"
    return dict(missing=missing, loaded=loaded, worst=worst, table_shape=list(msd[tbl].shape),
                init_params_equal=sorted(set(ref.init_params)) == sorted(set(mine.init_params)),
                init_params_ref=len(set(ref.init_params)), has_lm_cap=any("lm_cap_head" in n for n in mine.init_params))


def _ref_module(name):
    spec = importlib.util.spec_from_file_location("models." + name, os.path.join(REF, "models", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["models." + name] = mod
    spec.loader.exec_module(mod)
    return mod


def subclass():
    import xfm_b200.xfm as X
    pkg = types.ModuleType("models")
    pkg.__path__ = [os.path.join(REF, "models")]
    pkg.XFMBase, pkg.build_mlp, pkg.load_pretrained = X.XFMBase, X.build_mlp, X.load_pretrained
    sys.modules["models"], sys.modules["models.xfm"] = pkg, X
    cfg = O.tiny_config()
    tdir, vckpt = synth_checkpoints(cfg, src_window=4)
    config = our_config(cfg, tdir, vckpt)
    out = {}

    # ---- Pretrain.py:413-417: PretrainModel(config=config); model.to(device)   (defaults: both load_*_params True)
    XFM = _ref_module("model_pretrain").XFM
    model = XFM(config=config)
    model = model.to(torch.device("cpu"))
    out["pretrain_is_ours"] = isinstance(model, X.XFMBase) and XFM.__module__ == "models.model_pretrain"
    want = set(O.expand_tied(O.make_state_dict(cfg), cfg))
    out["pretrain_missing_keys"] = sorted(want - set(model.state_dict()))[:5]
    B, Lt, N, D = 3, 8, model._vis.N, model.vision_width
    calls = []

    def rec(name, ret):
        def f(*a, **k):
            calls.append((name, sorted(k)))
            return ret(*a, **k) if callable(ret) else ret
        return f
    one = lambda: torch.ones((), requires_grad=True) * 1.0
    model.get_vision_embeds = rec("vision", lambda image, image_atts=None, idx_to_group_img=None, do_mask=False:
                                  (torch.zeros(B, N, D), torch.ones(B, N, dtype=torch.long)) + ((torch.zeros(B, N - 1, dtype=torch.bool),) if do_mask else ()))
    model.get_text_embeds = rec("text", torch.zeros(B, Lt, model.text_width))
    model.get_features = rec("features", (torch.zeros(B, 4), torch.zeros(B, 4)))
    model.get_contrastive_loss = rec("itc", lambda *a, **k: one())
    model.get_matching_loss = rec("itm", lambda *a, **k: one())
    model.get_fuse_mlm_loss = rec("mlm", lambda *a, **k: one())
    model.get_mim_loss = rec("mim", lambda *a, **k: one())
    with torch.no_grad():
        model.temp.fill_(0.9)
    v0 = model.flat.P._version
    res = model(torch.zeros(B, 3, 64, 64), torch.zeros(B, Lt, dtype=torch.long), torch.ones(B, Lt, dtype=torch.long),
                text_ids_masked=torch.zeros(B, Lt, dtype=torch.long), masked_pos=torch.zeros(B, 2, dtype=torch.long),
                masked_ids=torch.zeros(B, 2, dtype=torch.long), ret_mim_loss=True, data_source="image")
    out["forward_keys"] = sorted(res)
    out["forward_calls"] = [c[0] for c in calls]
    out["itm_kwargs"] = [c[1] for c in calls if c[0] == "itm"][0]
    out["temp_after_clamp"] = float(model.temp)                       # model_pretrain.py:35-37 ran on our parameter
    out["master_version_unchanged"] = model.flat.P._version == v0     # ... without looking like an edit of the flat buffer
    out["temp_in_flat"] = float(model.flat.view32("temp"))
    txt = model.forward_text.__func__ is XFM.forward_text
    out["forward_text_is_reference"] = bool(txt)

    # ---- the optimizer / scheduler / accelerator sequence of Pretrain.py:426-447 on the host
    from xfm_b200.accelerator import B200DDPAccelerator, FlatAdamW
    opt = FlatAdamW(model, lr=1e-4, weight_decay=0.01, lr_mult=2)
    torch.optim.lr_scheduler.LambdaLR(opt, lambda s: 1.0)
    acc = B200DDPAccelerator(types.SimpleNamespace(CLIP_GRAD_NORM=1.0, AUTO_CAST=False))
    wrapped, _, _ = acc.set_up(model, opt, None, 0, 1, 0)
    out["wrapped_module_is_model"] = wrapped.module is model

    # ---- model_retrieval.py / model_nlvr.py
    R = _ref_module("model_retrieval").XFMForRetrieval
    r = R(config=dict(config))
    out["retrieval_heads"] = r.num_attention_heads
    out["retrieval_init_params"] = r.init_params
    Nl = _ref_module("model_nlvr").XFMForNLVR
    n = Nl(config=dict(config)).to(torch.device("cpu"))
    out["nlvr_head_type"] = type(n.cls_head).__name__
    out["nlvr_init_params"] = n.init_params
    nopt = FlatAdamW(n, lr=1e-4, weight_decay=0.01, lr_mult=2)
    out["nlvr_head_adopted"] = sorted(n._extra_params)
    out["nlvr_large_lr_params"] = len(nopt.param_groups[2]["params"]) + len(nopt.param_groups[3]["params"])
    return out


if __name__ == "__main__":
    fn = {"loaders": loaders, "subclass": subclass}[sys.argv[1]]
    import contextlib
    import io
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        res = fn()
    print("PROBE_JSON " + json.dumps(res))
