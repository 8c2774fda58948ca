"""Import the UNMODIFIED reference (the XFM checkout named by XFM_REFERENCE_ROOT).  TEST INFRASTRUCTURE ONLY.

The reference pins transformers==4.12.5 / timm==0.4.12; this image has transformers 5.x and no timm.
The shim (SURVEY.md Appendix A) provides the handful of helpers the reference imports from those
packages; no reference source is copied or edited.  Only `tools/make_golden.py` and tests/ref_probe.py use
this module, and only where XFM_REFERENCE_ROOT names a checkout of the reference; the package never imports it.
"""
import importlib.machinery
import json
import math
import os
import sys
import tempfile
import types

import torch
import torch.nn as nn

REF_ROOT = os.environ.get("XFM_REFERENCE_ROOT", "")


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__spec__ = importlib.machinery.ModuleSpec(name, None)
    m.__path__ = []
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install():
    """Idempotent: registers stubs, patches transformers, puts the reference on sys.path."""
    if getattr(install, "_done", False):
        return
    if not os.path.isdir(REF_ROOT):
        raise RuntimeError(f"reference tree not found at {REF_ROOT}")
    import transformers  # noqa: F401  (must be imported before the timm stub exists)
    import transformers.modeling_utils as mu
    import transformers.pytorch_utils as pu

    mu.apply_chunking_to_forward = pu.apply_chunking_to_forward
    mu.prune_linear_layer = pu.prune_linear_layer

    def _no_prune(*a, **k):
        raise NotImplementedError

    mu.find_pruneable_heads_and_indices = _no_prune

    def get_head_mask(self, head_mask, n, *a, **k):
        assert head_mask is None
        return [None] * n

    mu.PreTrainedModel.get_head_mask = get_head_mask

    def init_weights(self):  # transformers 4.12.5 semantics: apply _init_weights, then tie embeddings
        self.apply(self._init_weights)
        out = self.get_output_embeddings() if hasattr(self, "get_output_embeddings") else None
        if out is not None and getattr(self.config, "tie_word_embeddings", True):
            out.weight = self.get_input_embeddings().weight

    mu.PreTrainedModel.init_weights = init_weights

    def drop_path(x, drop_prob: float = 0.0, training: bool = False):
        if drop_prob == 0.0 or not training:
            return x
        keep = 1 - drop_prob
        shape = (x.shape[0],) + (1,) * (x.ndim - 1)
        r = keep + torch.rand(shape, dtype=x.dtype, device=x.device)
        r.floor_()
        return x.div(keep) * r

    class DropPath(nn.Module):
        def __init__(self, drop_prob=None):
            super().__init__()
            self.drop_prob = drop_prob

        def forward(self, x):
            return drop_path(x, self.drop_prob, self.training)

    def to_2tuple(x):
        return tuple(x) if isinstance(x, (tuple, list)) else (x, x)

    _mod("timm")
    _mod("timm.models")
    _mod("timm.models.layers", drop_path=drop_path, DropPath=DropPath, to_2tuple=to_2tuple,
         trunc_normal_=torch.nn.init.trunc_normal_)
    _mod("timm.models.registry", register_model=lambda f: f)
    _mod("timm.models.vision_transformer", _cfg=lambda **k: dict(k), PatchEmbed=object)
    _mod("timm.models.helpers", load_pretrained=lambda *a, **k: None)
    _mod("timm.data")
    _mod("timm.data.constants", IMAGENET_DEFAULT_MEAN=(0.485, 0.456, 0.406), IMAGENET_DEFAULT_STD=(0.229, 0.224, 0.225),
         IMAGENET_INCEPTION_MEAN=(0.5, 0.5, 0.5), IMAGENET_INCEPTION_STD=(0.5, 0.5, 0.5))
    _mod("ftfy", fix_text=lambda s: s)
    import scipy.interpolate as _si

    # scipy >= 1.14 turned interp2d into a stub that raises (the reference's beit2.py:640 calls it).  On a rectilinear grid
    # interp2d(x, y, z, kind='cubic') is FITPACK regrid_smth with s=0 = RectBivariateSpline(y, x, z, kx=3, ky=3, s=0)
    # (scipy's interp2d migration guide).
    def interp2d(x, y, z, kind="cubic"):
        assert kind == "cubic"
        f = _si.RectBivariateSpline(y, x, z, kx=3, ky=3, s=0)
        return lambda xn, yn: f(yn, xn)

    _si.interp2d = interp2d
    sys.path.insert(0, REF_ROOT)
    import torch.distributed as dist

    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("gloo", rank=0, world_size=1)
    install._done = True


def roberta_config_dir(cfg):
    """Directory holding a roberta config.json with the dims in `cfg` (path must contain 'roberta')."""
    d = tempfile.mkdtemp(prefix="roberta-base-")
    js = dict(architectures=["RobertaForMaskedLM"], attention_probs_dropout_prob=cfg["attn_dropout"], bos_token_id=0,
              eos_token_id=2, hidden_act="gelu", hidden_dropout_prob=cfg["hidden_dropout"], hidden_size=cfg["hidden"],
              initializer_range=0.02, intermediate_size=cfg["ffn"], layer_norm_eps=cfg["ln_eps"],
              max_position_embeddings=cfg["max_pos"], model_type="roberta", num_attention_heads=cfg["heads"],
              num_hidden_layers=cfg["text_layers"], pad_token_id=cfg["pad_id"], type_vocab_size=cfg["type_vocab"],
              vocab_size=cfg["vocab_size"])
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump(js, f)
    return d


def bert_config_dir(cfg):
    """Directory holding a BERT config.json with the dims in `cfg` (path contains 'bert' and not 'roberta': xfm.py:260-265
    then builds models/xbert.py's BertForMaskedLM)."""
    d = tempfile.mkdtemp(prefix="bert-tiny-uncased-")
    js = dict(architectures=["BertForMaskedLM"], attention_probs_dropout_prob=cfg["attn_dropout"], hidden_act="gelu",
              hidden_dropout_prob=cfg["hidden_dropout"], hidden_size=cfg["hidden"], initializer_range=0.02,
              intermediate_size=cfg["ffn"], layer_norm_eps=cfg["ln_eps"], max_position_embeddings=cfg["max_pos"],
              model_type="bert", num_attention_heads=cfg["heads"], num_hidden_layers=cfg["text_layers"],
              pad_token_id=cfg["pad_id"], type_vocab_size=cfg["type_vocab"], vocab_size=cfg["vocab_size"])
    with open(os.path.join(d, "config.json"), "w") as f:
        json.dump(js, f)
    return d


def build_reference_xfm(cfg, sd_full, load_vision_params=False, load_text_params=False, vision_ckpt="", text_dir=None,
                        fp16_opt_level=None):
    """Build the reference's `models.model_pretrain.XFM` with dims from `cfg` and load `sd_full`
    (reference key layout, see oracle.xfm_oracle.expand_tied).  With sd_full None the model is returned as constructed;
    load_*_params / vision_ckpt / text_dir exercise the reference's constructor-time checkpoint import
    (models/xfm.py:205-256,298-385)."""
    install()
    import yaml

    cwd = os.getcwd()
    os.chdir(REF_ROOT)
    try:
        config = yaml.safe_load(open("configs/xfm-pt/Pretrain_XBrain_base_4m.yaml"))
        config["text_encoder"] = text_dir or (bert_config_dir(cfg) if cfg.get("text_arch") == "bert" else roberta_config_dir(cfg))
        if fp16_opt_level is not None:   # xfm.py:288-290: anything but 'O0' sets config_text.fp16 (xbert: scale q, not the scores)
            config["accelerator"] = dict(config.get("accelerator", {}), FP16_OPT_LEVEL=fp16_opt_level)
        config["image_res"] = cfg["image_res"]
        vdir = tempfile.mkdtemp(prefix="beit2-base-")
        with open(os.path.join(vdir, "config_beit2_base.json"), "w") as f:
            json.dump(dict(ckpt=vision_ckpt, vision_width=cfg["vision_width"], patch_size=cfg["patch_size"]), f)
        config["vision_config"] = os.path.join(vdir, "config_beit2_base.json")
        config["patch_size"] = cfg["patch_size"]
        config["text_num_hidden_layers"] = cfg["text_layers"]
        config["text_fusion_start_at"] = cfg["text_layers"]
        config["fusion_num_hidden_layers"] = cfg["fusion_layers"]
        config["embed_dim"] = cfg["embed_dim"]
        config["num_masking_patches"] = cfg["num_masking_patches"]
        config["min_num_patches"] = cfg["min_num_patches"]
        import models.beit2 as beit2
        import models.vqkd_vit as vqkd_vit  # noqa: F401
        import models.model_vqkd as model_vqkd
        from functools import partial

        orig_factory = beit2.beit_base_patch16
        orig_defaults = model_vqkd.get_model_default_params
        if cfg["vision_width"] != 768 or cfg["vision_depth"] != 12:
            # Same reference classes, smaller dims (the factory hard-codes ViT-B).  Forward code untouched.
            def small(img_size, **kw):
                return beit2.VisionTransformer(img_size=img_size, patch_size=cfg["patch_size"],
                                               embed_dim=cfg["vision_width"], depth=cfg["vision_depth"],
                                               num_heads=cfg["vision_heads"],
                                               mlp_ratio=cfg["vision_mlp"] / cfg["vision_width"],
                                               norm_layer=partial(nn.LayerNorm, eps=1e-6), **kw)

            beit2.beit_base_patch16 = small

            def small_defaults():
                d = orig_defaults()
                d.update(embed_dim=cfg["vision_width"], depth=cfg["vision_depth"], num_heads=cfg["vision_width"] // 64)
                return d

            model_vqkd.get_model_default_params = small_defaults
        if cfg["use_vision_tokenizer"]:
            # The tokenizer factory insists on a checkpoint file (model_vqkd.py:315-333): build the reference
            # VQKD once (teacher 'None'), overwrite encoder / task layer / codebook with the synthetic values.
            enc, dec = model_vqkd.get_model_default_params(), model_vqkd.get_model_default_params()
            enc.update(img_size=cfg["image_res"], num_classes=0)
            dec.update(img_size=cfg["image_res"] // dec["patch_size"], patch_size=1, in_chans=cfg["codebook_dim"],
                       num_classes=0, depth=3)
            vq = model_vqkd.VQKD(enc, dec, cfg["codebook_size"], cfg["codebook_dim"], teacher_model_type="None",
                                 decoder_out_dim=512, quantize_kmeans_init=False)
            vsd = vq.state_dict()
            n_over = 0
            for k, v in sd_full.items():
                if k.startswith("vqkd."):
                    kk = k[len("vqkd."):]
                    assert kk in vsd and tuple(vsd[kk].shape) == tuple(v.shape), (kk, v.shape)
                    vsd[kk] = v.clone()
                    n_over += 1
            assert n_over > 0
            vsd["quantize.embedding.initted"] = torch.Tensor([True])
            f = tempfile.NamedTemporaryFile(suffix=".pth", delete=False)
            torch.save({"model": vsd}, f.name)
            config.update(use_vision_tokenizer=True, tokenizer_model="vqkd_encoder_base_decoder_3x768x12_clip",
                          tokenizer_weight=f.name, codebook_size=cfg["codebook_size"], codebook_dim=cfg["codebook_dim"])
        try:
            from models.model_pretrain import XFM

            model = XFM(config, load_vision_params=load_vision_params, load_text_params=load_text_params)
        finally:
            beit2.beit_base_patch16 = orig_factory
            model_vqkd.get_model_default_params = orig_defaults
    finally:
        os.chdir(cwd)
    if sd_full is None:
        return model
    own = model.state_dict()
    load = {k: v for k, v in sd_full.items() if not k.startswith("vqkd.")}
    missing = [k for k in own if k not in load and not k.startswith("vqkd.")]
    unexpected = [k for k in load if k not in own]
    assert not missing, f"synthetic state_dict misses reference keys: {missing[:8]}"
    assert not unexpected, f"synthetic state_dict has keys the reference lacks: {unexpected[:8]}"
    for k, v in load.items():
        assert tuple(own[k].shape) == tuple(v.shape), (k, own[k].shape, v.shape)
    model.load_state_dict(load, strict=False)
    model.eval()
    return model


def build_reference_vqa(cfg, sd_full):
    """Build the reference's `models.model_generation.XFMForVQA` (BASELINE config #5) with dims from `cfg`
    (`dec_layers` decoder layers, decoder_fusion_start_at 0) and load `sd_full` (reference key layout)."""
    install()
    import contextlib
    import yaml

    if "dataset" not in sys.modules:
        # model_generation.py:17 imports build_tokenizer from the data package, which needs pycocotools etc.; XFMForVQA
        # never calls it.
        _mod("dataset", build_tokenizer=lambda *a, **k: None)
    cwd = os.getcwd()
    os.chdir(REF_ROOT)
    try:
        config = yaml.safe_load(open("configs/xfm-ft/VQA.yaml"))
        config["text_encoder"] = roberta_config_dir(cfg)
        config["image_res"] = cfg["image_res"]
        vdir = tempfile.mkdtemp(prefix="beit2-base-")
        with open(os.path.join(vdir, "config_beit2_base.json"), "w") as f:
            json.dump(dict(ckpt="", vision_width=cfg["vision_width"], patch_size=cfg["patch_size"]), f)
        config.update(vision_config=os.path.join(vdir, "config_beit2_base.json"), patch_size=cfg["patch_size"],
                      text_num_hidden_layers=cfg["text_layers"], text_fusion_start_at=cfg["text_layers"],
                      fusion_num_hidden_layers=cfg["fusion_layers"], num_dec_layers=cfg["dec_layers"],
                      decoder_fusion_start_at=0, pad_token_id=cfg["pad_id"])
        import models.beit2 as beit2
        from functools import partial

        orig_factory = beit2.beit_base_patch16
        if cfg["vision_width"] != 768 or cfg["vision_depth"] != 12:
            def small(img_size, **kw):
                return beit2.VisionTransformer(img_size=img_size, patch_size=cfg["patch_size"],
                                               embed_dim=cfg["vision_width"], depth=cfg["vision_depth"],
                                               num_heads=cfg["vision_heads"],
                                               mlp_ratio=cfg["vision_mlp"] / cfg["vision_width"],
                                               norm_layer=partial(nn.LayerNorm, eps=1e-6), **kw)

            beit2.beit_base_patch16 = small
        try:
            with contextlib.redirect_stdout(open(os.devnull, "w")):
                from models.model_generation import XFMForVQA

                model = XFMForVQA(config)
        finally:
            beit2.beit_base_patch16 = orig_factory
    finally:
        os.chdir(cwd)
    own = model.state_dict()
    # fine-tuning models hold a bare RobertaModel as text_encoder (xfm.py:397-403): keys lose the 'roberta.' level
    sd_full = {(k.replace("text_encoder.roberta.", "text_encoder.") if k.startswith("text_encoder.roberta.") else k): v
               for k, v in sd_full.items()}
    missing = [k for k in own if k not in sd_full]
    assert not missing, f"synthetic state_dict misses reference keys: {missing[:8]}"
    load = {k: v for k, v in sd_full.items() if k in own}
    for k, v in load.items():
        assert tuple(own[k].shape) == tuple(v.shape), (k, own[k].shape, v.shape)
    model.load_state_dict(load, strict=True)
    model.eval()
    return model
