"""text_classification.RobertaForSequenceClassification against transformers' RobertaForSequenceClassification (fp32, on the
CPU, eager) with the same random-init weights, in eval mode: logits, loss and every parameter gradient, for packed batches
(right padding of 1..128 tokens, masks with holes) and for the padded path a batch with a 200-token sequence takes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
tr = pytest.importorskip("transformers")

DIMS = dict(vocab_size=1000, hidden_size=256, num_hidden_layers=2, num_attention_heads=4, intermediate_size=1024,
            max_position_embeddings=260, hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
# every parameter gradient within this fraction of the parameter's largest |gradient| (bf16 GEMM operands and attention
# probabilities against fp32)
GRAD_TOL = 5e-2


def make(num_labels, seed=0, **over):
    from xfm_b200.text_classification import RobertaForSequenceClassification as M

    torch.manual_seed(seed)
    cfg = tr.RobertaConfig(num_labels=num_labels, **dict(DIMS, **over))
    ref = tr.RobertaForSequenceClassification(cfg).float().eval()
    mine = M(cfg)
    mine.load_state_dict(ref.state_dict())
    return ref, mine.to("cuda").eval()


def batch(lengths, Lpad, holes=False, seed=1):
    g = torch.Generator().manual_seed(seed)
    B = len(lengths)
    ids = torch.randint(3, DIMS["vocab_size"], (B, Lpad), generator=g)
    mask = torch.zeros((B, Lpad), dtype=torch.int64)
    for b, l in enumerate(lengths):
        mask[b, :l] = 1
        ids[b, l:] = 1   # pad_token_id
    ids[:, 0] = 0
    if holes:   # masked tokens inside the sequences (token 0 stays)
        hole = (torch.rand((B, Lpad), generator=g) < 0.2) & (torch.arange(Lpad) > 0)
        mask[hole] = 0
    return ids, mask


def compare(ref, mine, ids, mask, labels, record, tag):
    out_ref = ref(input_ids=ids, attention_mask=mask, labels=labels)
    out_ref.loss.backward()
    out = mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=labels.cuda())
    out.loss.backward()
    torch.cuda.synchronize()
    dlog = float((out.logits.detach().cpu() - out_ref.logits.detach()).abs().max())
    dloss = abs(float(out.loss.detach()) - float(out_ref.loss.detach())) / abs(float(out_ref.loss.detach()))
    gref = {n: p.grad for n, p in ref.named_parameters()}
    worst, worst_name = 0.0, None
    for n, p in mine.named_parameters():
        assert p.grad is not None, n
        g0 = gref[n]
        # a key bias shifts every score of a query row by the same amount: its exact gradient is zero, and what both sides
        # compute is rounding noise; it is bounded relative to the same layer's query-bias gradient instead
        scale = float(gref[n.replace("key.bias", "query.bias")].abs().max())
        if scale == 0.0:
            assert float(p.grad.abs().max()) == 0.0, n
            continue
        r = float((p.grad.cpu() - g0).abs().max()) / scale
        if r > worst:
            worst, worst_name = r, n
    record("text_classification", case=tag, logits_abs=dlog, loss_rel=dloss, grad_rel=worst, grad_worst=worst_name)
    print(tag, "logits", dlog, "loss", dloss, "grad", worst, worst_name)
    assert dlog <= 2e-2
    assert dloss <= 1e-3
    assert worst <= GRAD_TOL, (worst_name, worst)
    return out, out_ref


LENGTHS = [1, 2, 17, 40, 64, 65, 100, 127, 128, 5, 33, 90]


def test_ce_three_labels(record):
    ref, mine = make(3)
    ids, mask = batch(LENGTHS, 128)
    labels = torch.tensor([0, 1, 2] * 4)
    labels[3] = -100   # ignore_index
    out, _ = compare(ref, mine, ids, mask, labels, record, "ce3")
    assert out[0] is out.loss and out["logits"] is out.logits and out.logits.shape == (12, 3)


def test_mse_one_label(record):
    ref, mine = make(1, seed=3)
    ids, mask = batch(LENGTHS, 128, seed=4)
    compare(ref, mine, ids, mask, torch.linspace(0, 5, 12), record, "mse1")


def test_masks_with_holes(record):
    ref, mine = make(3, seed=5)
    ids, mask = batch(LENGTHS, 128, holes=True, seed=6)
    compare(ref, mine, ids, mask, torch.tensor([2, 1, 0] * 4), record, "holes")


def test_long_sequence_runs_padded(record):
    from xfm_b200 import lib as L

    ref, mine = make(3, seed=7)
    ids, mask = batch([200, 3, 50, 128], 200, seed=8)
    n0 = L.launch_count()
    compare(ref, mine, ids, mask, torch.tensor([0, 1, 2, 1]), record, "long200")
    assert L.launch_count() > n0


def test_optimizer_steps(record):
    """One torch.optim.AdamW step over model.parameters() on both sides: the logits still agree, so the bf16 shadow was
    recast from the updated fp32 buffer.  Both optimizers get this model's gradients: Adam's first step moves every
    element by about lr * sign(grad), so elements whose near-zero gradients differ in sign by rounding would otherwise
    move apart by 2 lr.  A FlatAdamW step runs too."""
    from xfm_b200.accelerator import FlatAdamW

    ref, mine = make(3, seed=9)
    ids, mask = batch(LENGTHS, 128, seed=10)
    labels = torch.tensor([0, 1, 2] * 4)
    before = mine(input_ids=ids.cuda(), attention_mask=mask.cuda()).logits.detach().cpu()
    opts = [torch.optim.AdamW(m.parameters(), lr=3e-3) for m in (ref, mine)]
    for model, opt, dev in ((ref, opts[0], "cpu"), (mine, opts[1], "cuda")):
        opt.zero_grad()
        model(input_ids=ids.to(dev), attention_mask=mask.to(dev), labels=labels.to(dev)).loss.backward()
    mg = dict(mine.named_parameters())
    with torch.no_grad():
        for n, p in ref.named_parameters():
            p.grad.copy_(mg[n].grad.cpu())
    for opt in opts:
        opt.step()
    after = mine(input_ids=ids.cuda(), attention_mask=mask.cuda()).logits.detach().cpu()
    want = ref(input_ids=ids, attention_mask=mask).logits.detach()
    moved = float((after - before).abs().max())
    err = float((after - want).abs().max())
    record("text_classification", case="adamw_step", moved=moved, logits_abs=err)
    assert moved > 0.05 and err <= 2e-2, (moved, err)
    opt = FlatAdamW(mine, lr=3e-3)
    opt.zero_grad()
    mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=labels.cuda()).loss.backward()
    opt.step()
    again = mine(input_ids=ids.cuda(), attention_mask=mask.cuda()).logits.detach().cpu()
    assert torch.isfinite(again).all() and float((again - after).abs().max()) > 1e-3


def test_train_mode_dropout():
    from xfm_b200 import lib as L

    ref, mine = make(3, seed=11, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    ids, mask = batch(LENGTHS, 128, seed=12)
    labels = torch.tensor([0, 1, 2] * 4).cuda()
    with torch.no_grad():
        ev = float(mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=labels).loss)
        mine.train()
        tr_loss = float(mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=labels).loss)
    assert tr_loss == ev
    _, mine = make(3, seed=11)
    mine.train()
    losses = []
    with torch.no_grad():
        for salt in (5, 5, 6):
            L.seed_salt_set(salt)
            mine._calls = 0
            losses.append(float(mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=labels).loss))
    L.seed_salt_set(0)
    assert losses[0] == losses[1] and losses[2] != losses[0], losses
    mine.eval()
    with torch.no_grad():
        ev = float(mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=labels).loss)
    assert ev != losses[0]


def test_rejects_invalid_inputs():
    _, mine = make(3)
    ids, mask = batch([5, 9], 16)
    bad = mask.clone()
    bad[1, 0] = 0
    with pytest.raises(ValueError, match="token 0"):
        mine(input_ids=ids.cuda(), attention_mask=bad.cuda())
    bad = mask.clone()
    bad[0] = 0
    with pytest.raises(ValueError, match="all-zero"):
        mine(input_ids=ids.cuda(), attention_mask=bad.cuda())
    with pytest.raises(ValueError, match="token_type_ids"):
        mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), token_type_ids=torch.ones_like(ids).cuda())
    out = mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), token_type_ids=torch.zeros_like(ids).cuda())
    assert out.loss is None and out[0] is out.logits
    with pytest.raises(NotImplementedError):
        mine(input_ids=ids.cuda(), attention_mask=mask.cuda(), labels=torch.zeros((2, 3)).cuda())
