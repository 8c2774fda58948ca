"""Timing of the ViT self-attention forward / backward on the tcgen05 key-block path: 577 tokens (384 px, W = 24) by default,
901 (480 px, W = 30) with N = 901.  usage: time_vit577.py [B] [N]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from xfm_b200 import lib as L  # noqa: E402

B, H, N = int(sys.argv[1]) if len(sys.argv) > 1 else 32, 12, int(sys.argv[2]) if len(sys.argv) > 2 else 577
W = int(round((N - 1) ** 0.5))
assert W * W + 1 == N, N
D = H * 64
g = torch.Generator(device="cuda").manual_seed(0)
qkv = torch.randn(B * N, 3 * D, device="cuda", generator=g).bfloat16()
table = torch.randn((2 * W - 1) ** 2 + 3, H, device="cuda", generator=g)
dout = torch.randn(B * N, D, device="cuda", generator=g).bfloat16()
dqkv = torch.empty_like(qkv)
ld = (N + 7) // 8 * 8
ds = torch.empty(B, H, N, ld, device="cuda", dtype=torch.bfloat16)
q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]


def fwd():
    return L.attention_fwd(q, k, v, B, H, N, N, 0.125, rel_table=table, rel_window=W)


def bwd(o, lse):
    L.attention_bwd(dout, q, k, v, o, lse, B, H, N, N, 0.125, dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:], ds_dump=ds,
                    rel_table=table, rel_window=W)


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1000 / n


o, lse = fwd()
fl = 4.0 * B * H * N * N * 64
uf, ub = timeit(fwd), timeit(lambda: bwd(o, lse))
print({"case": f"vit{N}", "B": B, "fwd_us": round(uf, 1), "bwd_us": round(ub, 1), "fwd_tflops": round(fl / uf / 1e6, 1),
       "bwd_tflops": round(2.5 * fl / ub / 1e6, 1)})
