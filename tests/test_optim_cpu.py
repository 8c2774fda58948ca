"""CPU checks of the optimizer half of the path (no GPU, no kernels):
  * the oracle restatement of transformers-4.12.5 AdamW + clip_grad_norm_ (oracle/optim_oracle.py) against torch's own Adam /
    clip_grad_norm_;
  * FlatAdamW's parameter-group membership for every parameter of the XFM layout against optim.py's rules — through the
    reference's own create_optimizer where XFM_REFERENCE_ROOT names a checkout of it, else the restated rule;
  * FlatAdamW is a torch.optim.Optimizer: scheduler.py's LambdaLR drives its param_groups and the values reach the
    hyper-parameter block the kernel reads."""
import importlib.util
import os
import sys

import pytest
import torch

from oracle import optim_oracle as OO
from oracle import xfm_oracle as O

REF = os.environ.get("XFM_REFERENCE_ROOT", "")


def test_oracle_adamw_against_torch_adam_and_clip():
    torch.manual_seed(0)
    p0 = torch.randn(257, 33)
    grads = [torch.randn(257, 33) * (0.1 + i) for i in range(4)]
    # weight_decay = 0: HF AdamW == torch Adam up to the placement of eps (eps vs eps * sqrt(1 - b2^t)): ~1e-8 / |g|
    p_ref = p0.clone().requires_grad_(True)
    adam = torch.optim.Adam([p_ref], lr=1e-3, betas=(0.9, 0.98), eps=1e-8)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for t, g in enumerate(grads, 1):
        p_ref.grad = g.clone()
        adam.step()
        OO.hf_adamw_step(p, g, m, v, t, 1e-3, 0.0, betas=(0.9, 0.98), eps=1e-8)
        torch.testing.assert_close(p, p_ref.detach(), rtol=1e-5, atol=1e-6)
    # decoupled decay is applied AFTER the Adam update with the plain lr: p <- p_adam * (1 - lr * wd)
    p2, m2, v2 = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    p3, m3, v3 = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    OO.hf_adamw_step(p2, grads[0], m2, v2, 1, 1e-3, 0.0)
    OO.hf_adamw_step(p3, grads[0], m3, v3, 1, 1e-3, 0.01)
    torch.testing.assert_close(p3, p2 * (1 - 1e-3 * 0.01), rtol=1e-6, atol=0)
    # clip_grad_norm_
    gs = [torch.randn(50, 7), torch.randn(300), torch.randn(3, 3, 3)]
    params = [torch.zeros_like(g).requires_grad_(True) for g in gs]
    for q, g in zip(params, gs):
        q.grad = g.clone()
    for max_norm in (0.5, 1e6):
        for q, g in zip(params, gs):
            q.grad = g.clone()
        total = torch.nn.utils.clip_grad_norm_(params, max_norm)
        mine_total, coef = OO.clip_grad_norm(gs, max_norm)
        torch.testing.assert_close(mine_total, total, rtol=1e-6, atol=0)
        for q, g in zip(params, gs):
            torch.testing.assert_close(g * coef, q.grad, rtol=1e-6, atol=0)


def _layout_model(**over):
    """The XFM-base LAYOUT (12 + 12 + 12 layers, every head, VQ-KD branch) at tiny widths: parameter names are those of
    the base model, which is all the grouping rules look at."""
    from xfm_b200.model_pretrain import XFM
    cfg = O.tiny_config(use_vision_tokenizer=True, vision_depth=12, text_layers=12, fusion_layers=12, **over)
    return XFM(dict(cfg), init=lambda n, s: torch.zeros(s), device="cpu"), cfg


def test_group_membership_matches_optim_py_rules():
    from xfm_b200.accelerator import FlatAdamW
    model, _ = _layout_model()
    opt = FlatAdamW(model, lr=1e-4, weight_decay=0.01, lr_mult=2.0)
    names = {id(p): n for n, p in model.named_parameters()}   # first name of tied parameters, like the reference sees them
    trainable = [n for n, p in model.named_parameters() if p.requires_grad]
    assert len(trainable) > 700
    want = {n: OO.group_of(n, set(model.init_params)) for n in trainable}
    have = {}
    for gi, g in enumerate(opt.param_groups):
        for p in g["params"]:
            have[names[id(p)]] = gi
    assert have == want
    hp = [(g["lr"], g["weight_decay"]) for g in opt.param_groups]
    assert hp == OO.group_hparams(1e-4, 0.01, 2.0)
    # spot checks of the substring rule (optim.py:17-25): every "...bias..." name, LayerNorm / norm weights -> no decay
    assert have["vision_encoder.blocks.3.attn.relative_position_bias_table"] == 1
    assert have["vision_encoder.blocks.3.attn.q_bias"] == 1 and have["vision_encoder.blocks.3.norm1.weight"] == 1
    assert have["vision_encoder.fc_norm.weight"] == 1   # "norm.weight" is a substring of "fc_norm.weight"
    assert have["text_encoder.lm_head.layer_norm.weight"] == 1   # "norm.weight" is a substring of "layer_norm.weight"
    assert have["itm_head.1.weight"] == 2                # the head's LayerNorm weight is named "1.weight": decays, large lr
    assert have["vision_encoder.blocks.3.gamma_1"] == 0 and have["temp"] == 2 and have["vision_proj.bias"] == 3
    assert not any(n.startswith("vqkd.") for n in have)  # frozen tokenizer


@pytest.mark.skipif(not os.path.isdir(REF), reason="XFM_REFERENCE_ROOT does not name a checkout of the original XFM sources")
def test_group_membership_through_the_reference_create_optimizer(monkeypatch):
    """optim.py:4-50 itself, with transformers.optimization.AdamW (removed in transformers 5) replaced by a recorder."""
    import types
    import transformers.optimization as topt
    monkeypatch.setattr(topt, "AdamW", lambda groups, **kw: groups, raising=False)
    spec = importlib.util.spec_from_file_location("_ref_optim", os.path.join(REF, "optim.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["_ref_optim"] = mod
    try:
        spec.loader.exec_module(mod)
    except NameError:
        pass   # optim.py:60 annotates with an undefined name further down (class LARS); create_optimizer is defined by then
    from xfm_b200.accelerator import FlatAdamW
    model, _ = _layout_model()
    groups = mod.create_optimizer(types.SimpleNamespace(lr=1e-4, weight_decay=0.01, lr_mult=2), model)
    opt = FlatAdamW(model, lr=1e-4, weight_decay=0.01, lr_mult=2)
    for gi in range(4):
        assert {id(p) for p in groups[gi]["params"]} == {id(p) for p in opt.param_groups[gi]["params"]}, gi
        assert groups[gi]["lr"] == opt.param_groups[gi]["lr"] and groups[gi]["weight_decay"] == opt.param_groups[gi]["weight_decay"]


def test_flat_adamw_is_a_torch_optimizer_driven_by_lambda_lr():
    from xfm_b200.accelerator import FlatAdamW
    from xfm_b200.model_pretrain import XFM
    model = XFM(dict(O.tiny_config()), init=lambda n, s: torch.zeros(s), device="cpu")
    opt = FlatAdamW(model, lr=2e-4, weight_decay=0.02, lr_mult=3.0)
    assert isinstance(opt, torch.optim.Optimizer)
    # scheduler.py:6-30: linear warm-up then linear decay through LambdaLR
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda step: min(1.0, (step + 1) / 4))
    assert [round(g["lr"] / g["initial_lr"], 6) for g in opt.param_groups] == [0.25] * 4
    hp = opt.hparams(max_grad_norm=1.0, grad_mul=0.5)
    torch.testing.assert_close(hp[:4], torch.tensor([5e-5, 5e-5, 1.5e-4, 1.5e-4]))
    torch.testing.assert_close(hp[4:8], torch.tensor([0.02, 0.0, 0.02, 0.0]))
    torch.testing.assert_close(hp[8:14], torch.tensor([0.9, 0.98, 1e-8, 1.0, 0.5, 1.0]))
    sd = opt.state_dict()
    assert set(sd) == {"state", "param_groups"} and sd["state"] == {}
    n_params = sum(len(g["params"]) for g in sd["param_groups"])
    assert n_params == sum(1 for p in model.parameters() if p.requires_grad)
    opt.load_state_dict(sd)
    assert sched.state_dict()["last_epoch"] == 0


def test_stray_parameters_are_adopted_into_a_flat_buffer():
    """model_nlvr.py:25 pattern: a build_mlp head assigned after XFMBase.__init__ (ordinary nn parameters)."""
    from xfm_b200.accelerator import FlatAdamW
    from xfm_b200.xfm import XFMBase, build_mlp

    class Nlvr(XFMBase):
        def __init__(self, config):
            super().__init__(config, device="cpu")
            self.cls_head = build_mlp(input_dim=self.text_width * 2, output_dim=2)
            self.init_params = ["cls_head." + n for n, _ in self.cls_head.named_parameters()]

    model = Nlvr(dict(O.tiny_config()))
    before = {n: p.detach().clone() for n, p in model.cls_head.named_parameters()}
    opt = FlatAdamW(model, lr=1e-4, weight_decay=0.01, lr_mult=2.0)
    assert model.flat_extra is not None and set(model._extra_params) == {"cls_head." + n for n in before}
    for n, p in model.cls_head.named_parameters():
        torch.testing.assert_close(p.detach(), before[n], rtol=0, atol=0)
        assert p.data_ptr() == model.flat_extra.view32("cls_head." + n).data_ptr()
        assert p.grad is not None and p.grad.data_ptr() == model.flat_extra._view(model.flat_extra.G, "cls_head." + n).data_ptr()
    in_groups = {id(p) for g in opt.param_groups for p in g["params"]}
    assert all(id(p) in in_groups for p in model.cls_head.parameters())
    assert len(opt.param_groups[2]["params"]) == 3 and len(opt.param_groups[3]["params"]) == 3   # large-lr groups
    # a driver that drops .grad (set_to_none) and lets autograd allocate a fresh one is folded back in
    w = model.cls_head[0].weight
    w.grad = None
    (w.sum() * 2).backward()
    model.collect_stray_grads()
    g = model.flat_extra._view(model.flat_extra.G, "cls_head.0.weight")
    assert w.grad.data_ptr() == g.data_ptr() and float(g.mean()) == 2.0
    model.zero_grad()
    assert float(g.abs().sum()) == 0.0 and w.grad.data_ptr() == g.data_ptr()


def test_create_scheduler_matches_reference_schedule():
    """xfm_b200.accelerator.create_scheduler against scheduler.py:4-32 run by tools/make_golden_feed.py: the learning rates
    of a two-group optimizer over the whole schedule (float and int warm-up, zero warm-up, past the end) and the values the
    reference writes back into args."""
    import json
    from xfm_b200.accelerator import create_scheduler

    class AttrDict(dict):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.__dict__ = self

    with open(os.path.join(os.path.dirname(__file__), "golden", "feed.json")) as f:
        cases = json.load(f)["scheduler"]
    assert len(cases) == 4
    for g in cases:
        args = AttrDict(dict(g["args"]))
        opt = torch.optim.SGD([dict(params=[torch.nn.Parameter(torch.zeros(1))], lr=1e-4),
                               dict(params=[torch.nn.Parameter(torch.zeros(1))], lr=2e-4)], lr=1e-4)
        sch = create_scheduler(args, opt)
        assert [args["num_training_steps"], args["num_warmup_steps"]] == g["resolved"]
        lrs = []
        for _ in range(args["num_training_steps"] + 3):
            lrs.append([grp["lr"] for grp in opt.param_groups])
            opt.step()
            sch.step()
        assert lrs == g["lrs"], g["args"]
    with pytest.raises(NotImplementedError):
        create_scheduler(AttrDict(sched="cosine", num_training_steps=4, num_warmup_steps=1), opt)


def test_create_optimizer_mirrors_optim_py_factory():
    """create_optimizer(args, model) (optim.py:4-50): lr / weight_decay / optional lr_mult from args, betas (0.9, 0.98), eps 1e-8."""
    import types
    from xfm_b200.accelerator import FlatAdamW, create_optimizer
    from xfm_b200.model_pretrain import XFM
    model = XFM(dict(O.tiny_config()), init=lambda n, s: torch.zeros(s), device="cpu")
    opt = create_optimizer(types.SimpleNamespace(lr=3e-4, weight_decay=0.05, lr_mult=2), model)
    assert isinstance(opt, FlatAdamW)
    assert [g["lr"] for g in opt.param_groups] == [3e-4, 3e-4, 6e-4, 6e-4]
    assert [g["weight_decay"] for g in opt.param_groups] == [0.05, 0.0, 0.05, 0.0]
    hp = opt.hparams(max_grad_norm=1.0, grad_mul=1.0)
    torch.testing.assert_close(hp[8:11], torch.tensor([0.9, 0.98, 1e-8]))
    plain = create_optimizer(types.SimpleNamespace(lr=1e-4, weight_decay=0.01), XFM(dict(O.tiny_config()), init=lambda n, s: torch.zeros(s), device="cpu"))
    assert [g["lr"] for g in plain.param_groups] == [1e-4] * 4          # lr_mult defaults to 1
