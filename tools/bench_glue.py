"""Time of an MNLI-shaped fine-tuning step on one GPU: RobertaForSequenceClassification (roberta-base dimensions, 3 labels,
random init, synthetic tokens) forward + backward + AdamW at batch 32 and max_seq_length 128.

    python tools/bench_glue.py --out DIR [--steps 20 --warmup 5 --batch 32 --max-len 128 --iters 200]

Two length mixes: "ragged" (a seeded uniform mix of 8..128 tokens per sequence, right padded to 128) and "full" (every
sequence 128 tokens).  For each mix:
  xfm_b200           this package (packed variable-length encoder, FlatAdamW)
  hf_bf16 / hf_fp32  transformers' RobertaForSequenceClassification in eager PyTorch on the same GPU (torch.optim.AdamW),
                     under bf16 autocast and in fp32
and, at kernel level (CUDA events over --iters launches of each), the packed attention (xfm_attention_varlen_fwd / _bwd)
against lib.attention_fwd / attention_bwd (mma.sync kernels) on the padded [32, 128] layout with a key mask, 12 heads.
Step times come from CUDA events around --steps steps after --warmup untimed ones.  The algorithmic FLOPs are counted
from the shapes (real tokens only, forward + backward = 3x forward; attention over each sequence's own keys).  The card
name and power limit are read in the same run.  Writes DIR/glue.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

D, H, NL, FF, LAYERS, VOCAB = 768, 12, 3, 3072, 12, 50265


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def mix_lengths(kind, B, Lmax, seed):
    if kind == "full":
        return [Lmax] * B
    rng = np.random.default_rng(seed)
    return rng.integers(8, Lmax + 1, B).tolist()


def make_batch(lengths, Lmax, dev, seed):
    g = torch.Generator().manual_seed(seed)
    B = len(lengths)
    ids = torch.randint(3, VOCAB - 1, (B, Lmax), generator=g)
    ids[:, 0] = 0
    mask = torch.zeros((B, Lmax), dtype=torch.int64)
    for b, l in enumerate(lengths):
        mask[b, :l] = 1
        ids[b, l:] = 1
    labels = torch.randint(0, NL, (B,), generator=g)
    return ids.to(dev), mask.to(dev), labels.to(dev)


def flops(lengths):
    """Forward + backward (3x forward) algorithmic FLOPs of the encoder and head on the real tokens."""
    T = sum(lengths)
    per_layer = 2 * T * D * (3 * D + D + 2 * FF) + sum(4 * l * l * D for l in lengths)
    head = 2 * len(lengths) * D * (D + NL)
    return 3 * (LAYERS * per_layer + head)


def time_steps(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bench_models(lengths, a, dev, out):
    from transformers import RobertaConfig
    from transformers import RobertaForSequenceClassification as HF

    from xfm_b200.accelerator import FlatAdamW
    from xfm_b200.text_classification import RobertaForSequenceClassification as M

    cfg = RobertaConfig(vocab_size=VOCAB, hidden_size=D, num_hidden_layers=LAYERS, num_attention_heads=H, intermediate_size=FF,
                        max_position_embeddings=514, type_vocab_size=1, layer_norm_eps=1e-5, num_labels=NL)
    ids, mask, labels = make_batch(lengths, a.max_len, dev, 3)
    model = M(cfg).to(dev).train()
    opt = FlatAdamW(model, lr=2e-5, weight_decay=0.01)

    def step_mine():
        opt.zero_grad()
        model(input_ids=ids, attention_mask=mask, labels=labels).loss.backward()
        opt.step()
    out["xfm_b200"] = time_steps(step_mine, a.steps, a.warmup)
    del model, opt
    torch.cuda.empty_cache()
    hf = HF(cfg).to(dev).train()
    hopt = torch.optim.AdamW(hf.parameters(), lr=2e-5, weight_decay=0.01)
    for name, amp in (("hf_bf16", True), ("hf_fp32", False)):
        def step_hf():
            hopt.zero_grad()
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
                loss = hf(input_ids=ids, attention_mask=mask, labels=labels).loss
            loss.backward()
            hopt.step()
        out[name] = time_steps(step_hf, a.steps, a.warmup)
    del hf, hopt
    torch.cuda.empty_cache()


def bench_attention(lengths, a, dev, out):
    from xfm_b200 import lib as L

    B, Lp, W = len(lengths), a.max_len, H * 64
    g = torch.Generator(device=dev).manual_seed(5)
    T = sum(lengths)
    qkv = torch.randn((T, 3 * W), generator=g, device=dev).to(torch.bfloat16)
    dout = torch.randn((T, W), generator=g, device=dev).to(torch.bfloat16)
    cu, tiles = L.varlen_plan(lengths)
    cu, tiles = cu.to(dev), tiles.to(dev)
    real = torch.cat([torch.arange(b * Lp, b * Lp + l) for b, l in enumerate(lengths)]).to(dev)
    qkv_p = torch.zeros((B * Lp, 3 * W), dtype=torch.bfloat16, device=dev)
    qkv_p[real] = qkv
    dout_p = torch.zeros((B * Lp, W), dtype=torch.bfloat16, device=dev)
    dout_p[real] = dout
    kmask = torch.full((B, Lp), -10000.0, device=dev)
    kmask.view(-1)[real] = 0.0
    dq = torch.empty_like(qkv)
    dq_p = torch.empty_like(qkv_p)
    sl = lambda t: (t[:, :W], t[:, W:2 * W], t[:, 2 * W:])
    o, lse = L.attention_varlen_fwd(*sl(qkv), cu, tiles, H, Lp, 0.125, dropout_p=0.1, dropout_seed=1)
    op, lsep = L.attention_fwd(*sl(qkv_p), B, H, Lp, Lp, 0.125, kmask=kmask, dropout_p=0.1, dropout_seed=1)
    runs = dict(
        varlen_fwd=lambda: L.attention_varlen_fwd(*sl(qkv), cu, tiles, H, Lp, 0.125, dropout_p=0.1, dropout_seed=1, out=o),
        varlen_bwd=lambda: L.attention_varlen_bwd(dout, *sl(qkv), o, lse, cu, tiles, H, Lp, 0.125, *sl(dq), dropout_p=0.1,
                                                  dropout_seed=1),
        padded_fwd=lambda: L.attention_fwd(*sl(qkv_p), B, H, Lp, Lp, 0.125, kmask=kmask, dropout_p=0.1, dropout_seed=1, out=op),
        padded_bwd=lambda: L.attention_bwd(dout_p, *sl(qkv_p), op, lsep, B, H, Lp, Lp, 0.125, *sl(dq_p), kmask=kmask,
                                           dropout_p=0.1, dropout_seed=1))
    res = {}
    for name, fn in runs.items():
        res[name + "_us"] = time_steps(fn, a.iters, 10) * 1000.0
    res["attention_flops_fwd"] = sum(4 * l * l * W for l in lengths)
    out["attention"] = res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--max-len", type=int, default=128)
    ap.add_argument("--iters", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_glue.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    from xfm_b200 import lib as L
    L.lib()
    result = dict(card=card(), batch=a.batch, max_seq_length=a.max_len, steps=a.steps, warmup=a.warmup, mixes={})
    for kind in ("ragged", "full"):
        lengths = mix_lengths(kind, a.batch, a.max_len, 17)
        r = dict(tokens=sum(lengths), padding_fraction=1.0 - sum(lengths) / (a.batch * a.max_len), step_flops=flops(lengths))
        ms = {}
        bench_models(lengths, a, dev, ms)
        r["ms_per_step"] = ms
        r["sequences_per_s"] = {k: a.batch / (v / 1000.0) for k, v in ms.items()}
        r["achieved_tflops"] = {k: r["step_flops"] / (v / 1000.0) / 1e12 for k, v in ms.items()}
        bench_attention(lengths, a, dev, r)
        result["mixes"][kind] = r
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "glue.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
