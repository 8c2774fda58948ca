"""The drop-in boundary, checked on the host (no kernels run):
  * constructor-time checkpoint import (load_vision_params / load_text_params, models/xfm.py:205-256,298-385 and
    models/beit2.py:572-673) equals the reference's own loaders on the same synthetic checkpoints;
  * the reference's OWN models/model_pretrain.py, model_retrieval.py and model_nlvr.py source subclasses xfm_b200.XFMBase
    unchanged: the Pretrain.py:413-417 construction sequence, forward_multimodal's call pattern, temp.clamp_, the
    optimizer / accelerator set-up;
  * relative-position table resampling (models/beit2.py:611-652) properties.
The two reference-dependent checks run tests/ref_probe.py in a subprocess and are skipped unless XFM_REFERENCE_ROOT names a
checkout of the original XFM sources."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("XFM_REFERENCE_ROOT", "")
needs_ref = pytest.mark.skipif(not os.path.isdir(REF),
                               reason="XFM_REFERENCE_ROOT does not name a checkout of the original XFM sources")


def _probe(mode):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "ref_probe.py"), mode], capture_output=True, text=True,
                       timeout=600, env=dict(os.environ, MASTER_PORT="29577"))
    lines = [l for l in r.stdout.splitlines() if l.startswith("PROBE_JSON ")]
    assert r.returncode == 0 and lines, r.stderr[-3000:]
    return json.loads(lines[-1][len("PROBE_JSON "):])


@needs_ref
def test_constructor_checkpoint_import_equals_the_reference_loaders():
    res = _probe("loaders")
    assert res["missing"] == []
    assert res["loaded"] >= 80 and res["worst"] <= 1e-6, res        # every vision / text tensor, incl. the resampled tables
    assert res["table_shape"] == [52, 2]                              # 6x6-window checkpoint -> 4x4-window model
    assert res["init_params_equal"] and res["init_params_ref"] == 23 and res["has_lm_cap"]


@needs_ref
def test_reference_task_model_sources_run_on_xfm_b200():
    res = _probe("subclass")
    assert res["pretrain_is_ours"] and res["pretrain_missing_keys"] == []
    assert res["forward_keys"] == ["loss_bbox", "loss_giou", "loss_itc", "loss_itm", "loss_mim", "loss_mlm"]
    assert res["forward_calls"] == ["vision", "text", "features", "itc", "itm", "mlm", "vision", "mim"]
    assert res["itm_kwargs"] == ["text_embeds"]
    assert res["temp_after_clamp"] == 0.5 and res["temp_in_flat"] == 0.5 and res["master_version_unchanged"]
    assert res["forward_text_is_reference"] and res["wrapped_module_is_model"]
    assert res["retrieval_heads"] == 2 and res["retrieval_init_params"] == []
    assert res["nlvr_head_type"] == "_Mlp" and len(res["nlvr_init_params"]) == 6
    assert len(res["nlvr_head_adopted"]) == 6 and res["nlvr_large_lr_params"] == 6


def test_relative_position_table_resampling_properties():
    from xfm_b200.checkpoint import interpolate_rel_pos
    torch.manual_seed(0)
    H, src = 3, 13   # 7x7 window -> 13 offsets per axis
    tab = torch.randn(src * src + 3, H)
    assert interpolate_rel_pos(tab, src) is tab                       # same size: untouched (beit2.py:624)
    for dst in (27, 7):                                                # 14x14 (224 px) and 4x4 windows
        out = interpolate_rel_pos(tab, dst)
        assert out.shape == (dst * dst + 3, H) and out.dtype == torch.float32
        torch.testing.assert_close(out[-3:], tab[-3:])                # the three cls entries are carried over
        # the centre offset (0, 0) is a knot of both grids: value preserved
        torch.testing.assert_close(out[(dst * dst) // 2], tab[(src * src) // 2], rtol=1e-5, atol=1e-5)
    # an interpolating bicubic spline reproduces cubic polynomials: sample one on the reference's geometric source grid
    # (beit2.py:629-655) and compare on the integer target grid
    dst = 27
    left, right = 1.01, 1.5
    while right - left > 1e-6:
        q = (left + right) / 2.0
        gp = (1.0 - q ** (src // 2)) / (1.0 - q)
        right, left = (q, left) if gp > dst // 2 else (right, q)
    dis, cur = [], 1
    for i in range(src // 2):
        dis.append(cur)
        cur += q ** (i + 1)
    x = torch.tensor([-d for d in reversed(dis)] + [0] + dis, dtype=torch.float64)
    poly = lambda yy, xx: 0.3 + 0.02 * xx - 0.01 * yy + 1e-3 * xx * yy + 2e-4 * xx ** 3 - 1e-4 * yy ** 2 * xx
    z = poly(x[:, None], x[None, :]).reshape(-1, 1).float()
    tab = torch.cat([z, torch.zeros(3, 1)])
    out = interpolate_rel_pos(tab, dst)[:-3].reshape(dst, dst).double()
    t = torch.arange(-(dst // 2), dst // 2 + 1, dtype=torch.float64)
    torch.testing.assert_close(out, poly(t[:, None], t[None, :]), rtol=1e-4, atol=1e-4)


def test_host_construction_then_to_device_sequence_without_a_gpu():
    """Pretrain.py:413-417 on a GPU-less host: construct, .to(cpu) is a no-op, state_dict round trip, fp16 refused."""
    from oracle import xfm_oracle as O
    from xfm_b200.model_pretrain import XFM
    cfg = O.tiny_config(use_vision_tokenizer=True)
    model = XFM(dict(cfg), init=lambda n, s: O.make_tensor(n, s, 0))
    assert model.flat.P.device.type == ("cuda" if torch.cuda.is_available() else "cpu")
    assert model.to(model.flat.P.device) is model
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    model.load_state_dict(sd)
    with pytest.raises(RuntimeError, match="fp32 master"):
        model.half()
    # learnable_temp False: temp is a python float and not a state_dict entry (xfm.py:505-507)
    frozen = XFM(dict(cfg, learnable_temp=False), init=lambda n, s: O.make_tensor(n, s, 0))
    assert isinstance(frozen.temp, float) and "temp" not in frozen.state_dict() and "temp" not in frozen.init_params


def test_unbuilt_configurations_are_rejected_loudly():
    """Layouts the reference supports but this package does not build must fail at construction, never run as something
    else: local vision attention (beit2.py forward_localattn), CLIP / Swin vision encoders, text-side cross-attention."""
    import pytest
    from xfm_b200.config import normalize_config
    base = dict(text_num_hidden_layers=2, fusion_num_hidden_layers=2)
    normalize_config(dict(base, local_attn_depth=-1))
    for bad in (dict(local_attn_depth=2), dict(use_beit_v2=False), dict(text_fusion_start_at=1), dict(fusion_fusion_start_at=1)):
        with pytest.raises(NotImplementedError):
            normalize_config(dict(base, **bad))


def test_base_class_load_pretrained_resamples_for_a_larger_resolution(tmp_path):
    """XFMBase.load_pretrained (xfm.py:542-557), the call Retrieval.py / NLVR.py make on a 224-px pre-training checkpoint with a
    384-px model: here 64 px -> 96 px on the tiny layout.  Vision tables are resampled (beit2.py:753-808), every other weight
    arrives unchanged, text keys of a bare-encoder checkpoint land on this module's layout."""
    from oracle import xfm_oracle as O
    from xfm_b200 import checkpoint as CK
    from xfm_b200.model_pretrain import XFM
    cfg = O.tiny_config(use_vision_tokenizer=False)
    src = XFM(dict(cfg), init=lambda n, s: O.make_tensor(n, s, 3))
    sd = {k: v.detach().clone() for k, v in src.state_dict().items()}
    path = str(tmp_path / "pt.th")
    torch.save({"model": sd}, path)
    cfg2 = dict(cfg, image_res=96)
    dst = XFM(dict(cfg2), init=lambda n, s: O.make_tensor(n, s, 5))
    dst.load_pretrained(path, dict(cfg2, use_beit_v2=True, text_encoder="roberta-base"))
    got = dst.state_dict()
    tab = [k for k in sd if k.endswith("relative_position_bias_table")]
    assert tab, "the tiny layout has relative-position tables"
    for k, v in sd.items():
        if k in tab:
            assert got[k].shape != v.shape
            want = CK.interpolate_rel_pos(v.cpu(), 2 * (96 // cfg["patch_size"]) - 1)
            assert torch.allclose(got[k].cpu(), want, atol=1e-6), k
        elif got[k].shape == v.shape:
            assert torch.equal(got[k].cpu(), v.cpu()), k
    assert torch.equal(got["text_encoder.roberta.encoder.layer.0.attention.self.query.weight"].cpu(),
                       sd["text_encoder.roberta.encoder.layer.0.attention.self.query.weight"].cpu())
