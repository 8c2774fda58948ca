#!/usr/bin/env python
"""bench.py — XFM-base pre-training step (ITC + ITM + MLM + MIM with VQ-KD targets) on synthetic 224 px / 40-token
batches (BASELINE.json configs[1]), one process per GPU.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps K --warmup W      # the reference algorithm on the host CPU cores
    python bench.py --steps K --warmup W --dump-outputs bench_outputs   # also write the last timed step's outputs (.npy)

One "step" = forward (vision x2, text x2, fusion over 4B pairs, VQ-KD tokenizer, heads) + backward + gradient
all-reduce + clip + AdamW on B pairs per GPU.  `value` is timed with the batches already resident in HBM; `e2e` repeats
the same K steps with each step's inputs copied from pinned host memory and the loss read back to the host inside the
timed region.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic FLOPs per image-text pair, fwd+bwd, measured on the reference with FlopCounterMode (SURVEY.md §8d):
# 406.94 GFLOP (ITC+ITM+MLM+MSE-MIM) + VQ-KD tokenizer fwd 35.47 + codebook 0.10 + lm_head 768->8192 on 75 rows 2.83
GFLOP_PER_PAIR = 445.3
# one fusion layer (self-attn + cross-attn over 197 image tokens + FFN), one sample-pass, L=40: 1.1545 GFLOP fwd, 3.46 fwd+bwd
# (SURVEY.md §8d); a pre-training pair makes 4 passes (pos, 2 hard negatives, MLM) through 12 layers
FUSION_GFLOP_PER_PAIR = 4 * 12 * 3.46
METRIC = "image-text pairs/sec/step"
UNIT = "pairs/s"
# 33 steps of the default workload (B = 96) take ~2.1 s on a B200 at 62-64 ms / step
WARMUP_MIN_STEPS = 33
# --dump-outputs: size of the fixed, seeded sample of the fp32 master weights written after the dumped step (16 MB)
DUMP_PARAM_SAMPLES = 1 << 22


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region through NVML (the same counters the
    `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` line of B200_PROFILING.md prints).  NVML calls release the
    GIL and take microseconds; forking nvidia-smi from a thread stalled the launching thread for tens of ms per step."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.bits, self.max_mhz, self._stop_evt = index, [], 0, None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        while not self._stop_evt.is_set():
            try:
                self.sm.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                try:
                    self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            self._stop_evt.wait(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": [n for bit, n in self.REASONS.items() if self.bits & bit], "samples": len(sm), "source": "nvml"}


# ----------------------------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY.md §8d config #2)
# ----------------------------------------------------------------------------------------------------------------------
def base_config():
    return dict(image_res=224, patch_size=16, use_vision_tokenizer=True, codebook_size=8192, codebook_dim=32, embed_dim=256,
                temp=0.07, num_masking_patches=75, min_num_patches=16, use_bbox=True)


def gpu_init(device, seed):
    """Random-init weights of the XFM-base architecture, generated on the device (O(1) activations through depth)."""
    g = torch.Generator(device=device).manual_seed(seed)

    def init(name, shape):
        leaf = name.rsplit(".", 1)[-1]
        if name == "temp":
            return torch.tensor(0.07)
        if leaf in ("gamma_1", "gamma_2"):
            return torch.full(shape, 0.1, device=device)
        if ("norm" in name.lower() and leaf == "weight") or (name.endswith(".1.weight") and len(shape) == 1):
            return torch.ones(shape, device=device)
        if len(shape) <= 1 and leaf != "relative_position_bias_table":
            return 0.02 * torch.randn(shape, device=device, generator=g)
        if "quantize.embedding" in name:
            return torch.nn.functional.normalize(torch.randn(shape, device=device, generator=g), dim=-1)
        if "embeddings" in name or "pos_embed" in name or "patch_embed" in name or leaf == "relative_position_bias_table":
            return 0.05 * torch.randn(shape, device=device, generator=g)
        return (0.6 / shape[-1] ** 0.5) * torch.randn(shape, device=device, generator=g)
    return init


def make_host_batch(B, L, M, vocab, res, seed):
    g = torch.Generator().manual_seed(seed)
    image = torch.rand(B, 3, res, res, generator=g)
    ids = torch.randint(3, vocab - 1, (B, L), generator=g)
    ids[:, 0] = 0
    atts = torch.ones(B, L, dtype=torch.long)
    n_real = torch.randint(L // 2, L + 1, (B,), generator=g)
    ar = torch.arange(L).view(1, L)
    pad = ar >= n_real.view(B, 1)
    atts[pad] = 0
    ids[pad] = 1
    masked_pos = torch.zeros(B, M, dtype=torch.long)
    masked_ids = torch.full((B, M), -100, dtype=torch.long)
    ids_masked = ids.clone()
    for b in range(B):
        k = min(M, max(1, (int(n_real[b]) - 1) // 2))
        pos = torch.sort(torch.randperm(int(n_real[b]) - 1, generator=g)[:k] + 1).values
        masked_pos[b, :k] = pos
        masked_ids[b, :k] = ids[b, pos]
        ids_masked[b, pos] = vocab - 1
    out = dict(image=image, text_ids=ids, text_atts=atts, text_ids_masked=ids_masked, masked_pos=masked_pos, masked_ids=masked_ids)
    return {k: v.pin_memory() for k, v in out.items()}


LOSS_NAMES = ("loss_itc", "loss_itm", "loss_mlm", "loss_mim")


def step_outputs(loss, losses, norm, master):
    """What one training step hands its caller, as host float32 arrays: the loss, its four terms, the clipped gradient norm
    and the updated weights (a fixed, seeded sample of the flat fp32 master buffer)."""
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, master.numel(), (min(DUMP_PARAM_SAMPLES, master.numel()),), generator=g).sort().values
    out = dict(loss=loss, **losses, grad_norm=norm, params_sample=master[idx.to(master.device)])
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def _eager_legs(dev, B, steps, out):
    from oracle import xfm_oracle as O
    cfg = O.base_config(use_vision_tokenizer=True)
    init = gpu_init(dev, 0)
    shapes = dict(O.param_shapes(cfg))
    shapes.update(O.vqkd_param_shapes(cfg))
    sd = {k: init(k, s).to(dev) for k, s in shapes.items()}
    sd["temp"] = torch.tensor(0.07, device=dev)
    train = [v.requires_grad_(True) for k, v in sd.items() if not k.startswith("vqkd.") and v.dtype.is_floating_point]
    optim = torch.optim.AdamW(train, lr=1e-4, betas=(0.9, 0.98), eps=1e-8, weight_decay=0.01)
    batch = {k: v.to(dev) for k, v in O.make_batch(cfg, B, L=40, M=15, seed=1, image_uniform=True).items()}
    ineg, tneg = torch.roll(torch.arange(B, device=dev), 1), torch.roll(torch.arange(B, device=dev), -1)
    import random
    import numpy as np
    random.seed(1234)
    np.random.seed(1234)
    ids_mask = O.sample_mim_masks(cfg, B).to(dev)

    def step():
        res = O.pretrain_forward(sd, cfg, batch, ineg, tneg, ids_mask=ids_mask)
        loss = res["loss_itc"] + res["loss_itm"] + res["loss_mlm"] + res["loss_mim"]
        optim.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(train, 1.0)
        optim.step()
        return loss

    for name, autocast in (("bf16_autocast", True), ("fp32", False)):
        def run():
            if not autocast:
                return step()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return step()
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "loss": float(loss.detach())}
    out["peak_mem_gib"] = round(torch.cuda.max_memory_allocated(dev) / 2**30, 1)


def gpu_eager_baseline(dev, B, steps=3):
    """The comparator SURVEY.md §0.1 / §8d names: the reference algorithm as eager PyTorch library calls (cuBLAS / ATen
    kernels; oracle/xfm_oracle.py is that op sequence) on the SAME B200, same workload and batch, fwd + bwd + clip +
    torch.optim.AdamW, under bf16 autocast and in fp32.  Reported next to cpu_baseline; not the product path."""
    import gc
    out = {"pairs_per_step": B, "optimizer": "torch.optim.AdamW (foreach)", "steps": steps, "warmup": 1,
           "what": "oracle/xfm_oracle.py op sequence (= the reference's ATen calls) on cuda:0, eval-mode dropout"}
    try:
        _eager_legs(dev, B, steps, out)
    except Exception as e:  # an out-of-memory eager run is itself a result
        out["error"] = f"{type(e).__name__}: {str(e)[:200]}"
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    return out


def run_ours(args):
    import torch.distributed as dist
    from xfm_b200 import lib as L
    from xfm_b200.accelerator import B200DDPAccelerator, FlatAdamW, reserve_arena
    from xfm_b200.model_pretrain import XFM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # Exactly ONE JSON line may reach stdout.  NCCL prints its "NCCL version ..." banner with printf at NCCL_DEBUG=VERSION
    # (this image's default), so under torchrun file descriptor 1 is pointed at stderr for the whole run and the JSON line
    # goes to a private duplicate of the original stdout.
    out_stream = sys.stdout
    if world > 1:
        sys.stdout.flush()
        out_stream = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    wd = int(os.environ.get("XFM_BENCH_WATCHDOG", "0"))
    if wd > 0:   # debugging aid: dump every thread's stack to stderr if the run is still alive after `wd` seconds
        import faulthandler
        faulthandler.dump_traceback_later(wd, repeat=True, file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.graph:   # collectives inside a captured graph: torch's own guidance for NCCL + CUDA graphs
            os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        dist.init_process_group("nccl", device_id=dev)
    B, Lt, M = args.batch, 40, 15
    import random
    import numpy as np
    random.seed(1234 + rank)
    np.random.seed(1234 + rank)
    torch.manual_seed(1234 + rank)
    cfg = base_config()
    eager = None
    if world == 1 and rank == 0 and not args.no_eager:
        eager = gpu_eager_baseline(dev, B)
    model = XFM(cfg, init=gpu_init(dev, 0), device=dev).train()
    opt = FlatAdamW(model, lr=1e-4, weight_decay=0.01, lr_mult=2.0)
    acc = B200DDPAccelerator(dict(CLIP_GRAD_NORM=1.0, AUTO_CAST=False, OVERLAP_ALLREDUCE=args.overlap))
    wrapped, opt, _ = acc.set_up(model, opt, None, local, world, rank)
    n_pool = 4
    host = [make_host_batch(B, Lt, M, model.cfg["vocab_size"], 224, 100 + 17 * rank + i) for i in range(n_pool)]
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())

    def to_dev(hb):
        return {k: v.to(dev, non_blocking=True) for k, v in hb.items()}

    def step(b):
        out = wrapped(b["image"], b["text_ids"], b["text_atts"], text_ids_masked=b["text_ids_masked"], masked_pos=b["masked_pos"],
                      masked_ids=b["masked_ids"], ret_mim_loss=True, data_source="image")
        loss = out["loss_itc"] + out["loss_itm"] + out["loss_mlm"] + out["loss_mim"]
        acc.backward_step(loss, opt)
        norm = acc.optimizer_step(opt, wrapped)
        return loss.detach(), out, norm

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    resident = [to_dev(hb) for hb in host]
    i = 0
    # W warm-up steps, and at least WARMUP_MIN_STEPS: a GPU coming out of idle needs about a second under load before its
    # clocks and power state settle (first-loop timings varied by 15 % with 3 warm-up steps of 85 ms).  A fixed count, not
    # a time budget: every warm-up step updates the weights, so a count that followed the clock would make what the timed
    # steps compute depend on how fast the build is.
    n_warm = max(args.warmup, WARMUP_MIN_STEPS)
    while i < n_warm:
        loss, out, _ = step(resident[i % n_pool])
        if i == 0:
            arena = reserve_arena(factor=1.5)  # no cudaMalloc inside the timed regions (see accelerator.reserve_arena)
        if i % 4 == 3:
            torch.cuda.synchronize()
        i += 1
    warm_steps = i
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()

    step_stats = {}

    import gc

    def timed(fn, tag=None):
        # the cyclic garbage collector is run between the timed loops, not inside them: a generation-2 pass over the
        # ~10^5 live Python objects of this process takes 20-40 ms and starves the GPU for one step (step_ms max >> median)
        gc.collect()
        gc.disable()
        try:
            return _timed(fn, tag)
        finally:
            gc.enable()

    def _timed(fn, tag):
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        n0 = L.launch_count()
        evs[0].record()
        for i in range(args.steps):
            fn(i)
            evs[i + 1].record()
        barrier()
        ms = torch.tensor([evs[0].elapsed_time(evs[-1])], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if tag:   # per-step device times of this rank: a stall in one step shows as max >> median
            per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps))
            step_stats[tag] = {"min": per[0], "median": per[len(per) // 2], "max": per[-1]}
        return float(ms) / args.steps, L.launch_count() - n0

    last = {}

    def resident_step(i):
        last["loss"], last["out"], last["norm"] = step(resident[i % n_pool])

    # End-to-end loop: every step's inputs come from pinned host memory and its loss is read back.  The copy of step i+1 is
    # issued on a side stream while step i computes (what a prefetching loader does); both copies and the read-back are
    # inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    slots = [{k: torch.empty_like(v, device=dev) for k, v in host[0].items()} for _ in range(2)]  # static double buffer
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    staged = {"next": None}

    def stage(i):
        s = i & 1
        copy_stream.wait_event(consumed[s])  # the step that last used this slot has finished with it
        with torch.cuda.stream(copy_stream):
            for k, v in host[i % n_pool].items():
                slots[s][k].copy_(v, non_blocking=True)
            ready[s].record(copy_stream)
        staged["next"] = i

    def e2e_step(i):
        if staged["next"] != i:
            stage(i)
        s = i & 1
        torch.cuda.current_stream().wait_event(ready[s])
        stage(i + 1)
        loss, _, _ = step(slots[s])
        consumed[s].record(torch.cuda.current_stream())
        last["host_loss"] = float(loss.detach())  # D2H read of the step's result

    pairs_all = B * world
    ms_step, launches = timed(resident_step, "resident")
    dumped = None
    if args.dump_outputs and not args.graph:
        dumped = step_outputs(last["loss"], {k: last["out"][k] for k in LOSS_NAMES}, last["norm"], model.flat.P)
    ms_e2e, _ = timed(e2e_step, "e2e")
    graph_info = None
    if args.graph:   # the same step replayed as ONE CUDA graph (xfm_b200/graph.py)
        from xfm_b200.graph import GraphedStep

        def loss_fn(m, b):
            out = m(b["image"], b["text_ids"], b["text_atts"], text_ids_masked=b["text_ids_masked"], masked_pos=b["masked_pos"],
                    masked_ids=b["masked_ids"], ret_mim_loss=True, data_source="image")
            return (out["loss_itc"] + out["loss_itm"] + out["loss_mlm"] + out["loss_mim"],) + tuple(out[k] for k in LOSS_NAMES)
        gs = GraphedStep(wrapped, opt, acc, loss_fn, resident[0], warmup=3, uses_mim_masks=True)
        for i in range(3):
            gs(resident[i % n_pool])
        ms_g, _ = timed(lambda i: gs(resident[i % n_pool]), "graph_resident")
        if args.dump_outputs:   # gs.outputs = (loss, its four terms, gradient norm), overwritten by the next replay
            dumped = step_outputs(gs.outputs[0], dict(zip(LOSS_NAMES, gs.outputs[1:5])), gs.outputs[5], model.flat.P)

        g_staged = {"next": None}

        def g_e2e(i):   # inputs from pinned host memory (copy of step i+1 under step i, like a prefetching loader), loss read back
            if g_staged["next"] != i:
                gs.stage(host[i % n_pool])
            gs.commit()
            out = gs()                          # one graph launch; the host is free while the device runs the step
            gs.stage(host[(i + 1) % n_pool])    # next step's MIM masks sampled on the host + its H2D copy, under this step
            g_staged["next"] = i + 1
            last["host_loss"] = float(out[0])
        ms_ge, _ = timed(g_e2e, "graph_e2e")
        graph_info = {"ms_per_step": ms_g, "value": pairs_all / (ms_g * 1e-3), "e2e_ms_per_step": ms_ge,
                      "e2e_value": pairs_all / (ms_ge * 1e-3),
                      "unit": UNIT, "what": "forward + backward + clip + AdamW + zero_grad replayed as one CUDA graph"}
    clk = clocks.stop() if clocks else None

    # ---- fusion-layer leg: CUDA events around the 12 fusion layers (forward and backward of the 4B-sample pass) in three
    # steps issued back to back (the launch queue stays full, so the bracket holds kernel time, not host time); minimum.
    fus_ev = []

    def timed_call(fn):
        def wrapper(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            fus_ev.append((e0, e1))
            return r
        return wrapper
    fwd0, bwd0 = model._fus.layers_fwd, model._fus.layers_bwd
    model._fus.layers_fwd, model._fus.layers_bwd = timed_call(fwd0), timed_call(bwd0)
    gc.collect()
    gc.disable()
    n_fus = 3
    for i in range(n_fus):
        step(resident[i % n_pool])
    torch.cuda.synchronize()
    gc.enable()
    model._fus.layers_fwd, model._fus.layers_bwd = fwd0, bwd0
    per = len(fus_ev) // n_fus
    fus_ms = min(sum(a.elapsed_time(b) for a, b in fus_ev[i * per:(i + 1) * per]) for i in range(n_fus))
    # ---- roofline leg: one more step with CUDA events around every launch of the dominant kernel (the tcgen05 GEMM)
    L.gemm_profile = []
    step(resident[0])
    torch.cuda.synchronize()
    prof, L.gemm_profile = L.gemm_profile, None
    shapes = {}
    for p in prof:
        d = shapes.setdefault(p[3], [0, 0.0, 0.0])
        d[0] += 1
        d[1] += p[1].elapsed_time(p[2])
        d[2] += p[0]
    if rank == 0 and os.path.isdir(os.path.join(ROOT, "gpurun_out")):
        rows = [dict(M=k[0], N=k[1], K=k[2], a_t=k[3], b_t=k[4], count=v[0], ms=round(v[1], 4),
                     tflops=round(v[2] / (v[1] * 1e-3) / 1e12, 1) if v[1] > 0 else 0.0) for k, v in shapes.items()]
        rows.sort(key=lambda r: -r["ms"])
        with open(os.path.join(ROOT, "gpurun_out", "gemm_shapes.json"), "w") as f:
            json.dump(rows, f, indent=0)
    g_bytes = sum(p[4] for p in prof)
    g_flops = sum(p[0] for p in prof)
    g_ms = sum(p[1].elapsed_time(p[2]) for p in prof)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):  # dram__bytes_read + write per launch from the committed ncu --set full capture of this command
        with open(tpath) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    pk, pk_kind = peaks()
    peak = pk.get("bf16_tflops_sustained", 1400.0)
    ach = g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    losses = {k: float(v.detach()) for k, v in last["out"].items() if k in ("loss_itc", "loss_itm", "loss_mlm", "loss_mim")}

    pairs = B * world
    line = {
        "metric": METRIC, "value": pairs / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "warmup_steps_run": warm_steps, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic (uniform images, random token ids; random-init XFM-base weights)",
        "config": {"workload": "XFM-base pretraining step ITC+ITM+MLM+MIM(VQ-KD), 224px / 40 tokens / 15 masked, "
                               "fwd+bwd+allreduce+clip+AdamW", "pairs_per_gpu": B, "global_pairs": pairs,
                   "parallelism": f"dp{world}", "arena_gib": round(arena / 2**30, 1), "l2": "inputs and activations exceed L2 (>= 58 MB per activation tensor)",
                   "train_mode": True, "python_gc": "collected between the timed loops, disabled inside them"},
        "e2e": {"value": pairs / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                     "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram read+write, mean over every GEMM launch of a step)",
                     "algorithmic_bytes_per_launch": g_bytes / max(len(prof), 1),
                     "kernel": "gemm_tcgen05_pair_kernel / gemm_tcgen05_kernel", "launches_per_step": len(prof),
                     "gemm_ms_per_step": g_ms, "peak_source": f"{pk_kind} bf16_tflops_sustained",
                     "step_tflops_algorithmic": GFLOP_PER_PAIR * B / ms_step,
                     "step_frac_of_peak": GFLOP_PER_PAIR * B / ms_step / peak},
        "clocks": clk, "losses_last_step": losses, "step_ms": step_stats,
        # BASELINE.json's second figure: the 12 fusion layers (fwd + bwd of the 4B-sample pass), CUDA events around the
        # fusion encoder in one profiled step.  "algorithmic" counts the reference's FLOPs (K/V projection of an image
        # recomputed for each of its 4 passes); this implementation projects every image once per layer.
        "fusion_layer": {"ms_per_step": fus_ms, "tflops_algorithmic": FUSION_GFLOP_PER_PAIR * B / fus_ms if fus_ms > 0 else None,
                         "frac_of_peak": (FUSION_GFLOP_PER_PAIR * B / fus_ms / peak) if fus_ms > 0 else None,
                         "gflop_per_pair_algorithmic": FUSION_GFLOP_PER_PAIR, "peak": peak},
    }
    if eager is not None:
        line["gpu_eager_baseline"] = eager
    if graph_info is not None:
        # Headline = the step as the package's public API runs it for production (xfm_b200.graph.GraphedStep: the same
        # kernels, one graph launch per step); the launch-by-launch sequence is kept beside it.
        line["launch_sequence"] = {"value": line["value"], "ms_per_step": ms_step, "e2e_value": line["e2e"]["value"],
                                   "e2e_ms_per_step": ms_e2e, "unit": UNIT,
                                   "what": "the same step issued as individual kernel launches from Python (no graph)"}
        line["value"], line["ms_per_step"] = graph_info["value"], graph_info["ms_per_step"]
        line["e2e"].update(value=graph_info["e2e_value"], ms_per_step=graph_info["e2e_ms_per_step"])
        line["config"]["step"] = "one CUDA graph replay per step (forward + backward + all-reduce + clip + AdamW + zero_grad)"
        line["roofline"]["step_tflops_algorithmic"] = GFLOP_PER_PAIR * B / graph_info["ms_per_step"]
        line["roofline"]["step_frac_of_peak"] = GFLOP_PER_PAIR * B / graph_info["ms_per_step"] / peak
        line["graph_replays"] = args.steps
        line["cuda_graph"] = graph_info
    if rank == 0:
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args, quick=True)
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for k, v in dumped.items():
                np.save(os.path.join(args.dump_outputs, k + ".npy"), v)
        print(json.dumps(line), file=out_stream, flush=True)
    if world > 1:
        # leave without running destructors: tearing down a process group while captured graphs / side streams still
        # reference its communicator can block (seen with NCCL 2.28 after a graph capture)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stderr.flush()
        os._exit(0)


# ----------------------------------------------------------------------------------------------------------------------
# fine-tuning configurations (BASELINE configs[2..4]): --config retrieval | nlvr | vqa
# ----------------------------------------------------------------------------------------------------------------------
FINETUNE = {  # per-GPU batch, fwd+bwd GFLOP per sample at 384 px (SURVEY.md §8d), unit
    "retrieval": (32, 579.36, "pairs/s", "COCO-shape retrieval fine-tune (Retrieval_coco.yaml): ITC with idx soft labels + hard-negative ITM"),
    "nlvr": (64, 836.07, "texts/s", "NLVR2-shape fine-tune: two images per text through the fusion encoder"),
    "vqa": (24, 448.46, "questions/s", "VQA-shape fine-tune with the 12-layer causal answer decoder (3 answers x 8 tokens)"),
}


def finetune_workload(task, res, B, dev):
    """Model class + config, synthetic pinned host batches and the loss closure of one fine-tuning configuration."""
    import types
    B0, gflop, unit, what = FINETUNE[task]
    B = B or B0
    cfg = base_config()
    cfg.update(image_res=res, use_vision_tokenizer=False)
    if task == "retrieval":
        from xfm_b200.model_retrieval import XFMForRetrieval as Model
    elif task == "nlvr":
        from xfm_b200.model_nlvr import XFMForNLVR as Model
    else:
        from xfm_b200.model_generation import XFMForVQA as Model
        cfg.update(num_dec_layers=12, decoder_fusion_start_at=0, pad_token_id=1)
    torch.manual_seed(1234)
    g = torch.Generator().manual_seed(1)
    V, Lt, La, n_ans = 50265, 40, 8, 3

    def text(n, length, min_real):
        ids = torch.randint(3, V - 1, (n, length), generator=g)
        ids[:, 0] = 0
        n_real = torch.randint(min_real, length + 1, (n,), generator=g)
        pad = torch.arange(length).view(1, -1) >= n_real.view(-1, 1)
        atts = torch.ones(n, length, dtype=torch.long)
        atts[pad] = 0
        ids[pad] = 1
        return ids, atts

    n_img = 2 * B if task == "nlvr" else B
    host = [dict() for _ in range(2)]
    for hb in host:
        hb["image"] = torch.rand(n_img, 3, res, res, generator=g)
        hb["text_ids"], hb["text_atts"] = text(B, Lt, Lt // 2)
        if task == "retrieval":
            hb["idx"] = torch.randint(0, max(1, B // 5 * 4), (B,), generator=g)     # 5 captions per image => duplicates
        elif task == "nlvr":
            hb["targets"] = torch.randint(0, 2, (B,), generator=g)
        else:
            hb["a_ids"], hb["a_atts"] = text(B * n_ans, La, 3)
            hb["weights"] = torch.rand(B * n_ans, generator=g) * 0.8 + 0.2
    host = [{k: v.pin_memory() for k, v in hb.items()} for hb in host]
    k_dev = torch.full((B,), n_ans, dtype=torch.long, device=dev)

    def loss_fn(model, b):
        if task == "retrieval":
            l_itc, l_itm = model(b["image"], b["text_ids"], b["text_atts"], idx=b["idx"])
            return l_itc + l_itm
        if task == "nlvr":
            return model(b["image"], b["text_ids"], b["text_atts"], b["targets"])
        q = types.SimpleNamespace(input_ids=b["text_ids"], attention_mask=b["text_atts"])
        a = types.SimpleNamespace(input_ids=b["a_ids"], attention_mask=b["a_atts"])
        return model(b["image"], q, a, k=k_dev, weights=b["weights"], train=True)

    def build():
        from xfm_b200.accelerator import B200DDPAccelerator, FlatAdamW
        model = Model(cfg, init=gpu_init(dev, 0), device=dev).train()
        opt = FlatAdamW(model, lr=3e-5, weight_decay=0.01, lr_mult=2.0)
        acc = B200DDPAccelerator(dict(CLIP_GRAD_NORM=1.0))
        wrapped, opt, _ = acc.set_up(model, opt, None, 0, 1, 0)
        return model, wrapped, opt, acc
    return dict(B=B, n_img=n_img, gflop=gflop, unit=unit, what=what, host=host, loss_fn=loss_fn, build=build)


def run_finetune(args):
    """One process, one GPU: the fine-tuning step (forward + backward + clip + AdamW) of BASELINE configs #3-#5 at 384 px,
    timed as the eager launch sequence and as ONE replayed CUDA graph (xfm_b200/graph.py); `value` is the graph figure."""
    from xfm_b200 import lib as L
    from xfm_b200.graph import GraphedStep

    task = args.config
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    res = args.res
    wl = finetune_workload(task, res, args.batch if args.batch_given else 0, dev)
    B, n_img, gflop, unit, what, host, loss_fn, build = (wl[k] for k in ("B", "n_img", "gflop", "unit", "what", "host", "loss_fn", "build"))
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())

    def timed(fn, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = L.launch_count()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps, (L.launch_count() - n0) // steps

    resident = [{k: v.to(dev) for k, v in hb.items()} for hb in host]
    clocks = ClockSampler(dev.index or 0)
    # ---- eager launch sequence
    model, wrapped, opt, acc = build()

    def eager_step(i):
        loss = loss_fn(wrapped, resident[i & 1])
        acc.backward_step(loss, opt)
        acc.optimizer_step(opt, wrapped)
        return loss
    for i in range(max(args.warmup, 3)):
        eager_step(i)
    ms_eager, launches = timed(eager_step, args.steps)
    del model, wrapped, opt, acc
    torch.cuda.empty_cache()
    # ---- one CUDA graph per step
    model, wrapped, opt, acc = build()
    step = GraphedStep(wrapped, opt, acc, loss_fn, resident[0], warmup=max(args.warmup, 3))
    for i in range(3):
        step(resident[i & 1])
    clocks.start()
    ms_graph, _ = timed(lambda i: step(resident[i & 1]), args.steps)
    last = {}

    staged = {"next": None}

    def e2e_step(i):   # inputs from pinned host memory (copy of step i+1 issued under step i), loss read back, all timed
        if staged["next"] != i:
            step.stage(host[i & 1])
        step.commit()
        out = step()
        step.stage(host[(i + 1) & 1])
        staged["next"] = i + 1
        last["loss"] = float(out[0])
    ms_e2e, _ = timed(e2e_step, args.steps)
    clk = clocks.stop()
    pk, pk_kind = peaks()
    peak = pk.get("bf16_tflops_sustained", 1400.0)
    tfl = gflop * B / ms_graph if res == 384 else None
    line = {
        "metric": METRIC, "value": B / (ms_graph * 1e-3), "unit": unit, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_graph, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (uniform images, random token ids; random-init XFM-base weights)",
        "config": {"workload": what + f", {res} px / 40 tokens, fwd+bwd+clip+AdamW", "samples_per_gpu": B, "images_per_gpu": n_img,
                   "parallelism": "dp1", "train_mode": True, "step": "one CUDA graph replay (xfm_b200/graph.py)",
                   "l2": "activations exceed L2"},
        "e2e": {"value": B / (ms_e2e * 1e-3), "unit": unit, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
        "gpu_launches": launches * args.steps, "kernels_per_step": launches,
        "eager": {"value": B / (ms_eager * 1e-3), "unit": unit, "ms_per_step": ms_eager,
                  "what": "the same step as ~kernels_per_step individual launches from Python"},
        "roofline": {"bound": "tensor", "achieved": tfl, "peak": peak, "unit": "TFLOP/s", "frac": (tfl / peak) if tfl else None,
                     "traffic": None, "kernel": "whole step (algorithmic FLOPs of SURVEY.md §8d per sample)",
                     "peak_source": f"{pk_kind} bf16_tflops_sustained"},
        "clocks": clk, "loss_last_step": last.get("loss"),
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port, pinned to the reference's outputs by tests/test_oracle_golden.py)
# ----------------------------------------------------------------------------------------------------------------------
def _oracle_step_fn(B):
    from oracle import xfm_oracle as O
    torch.set_num_threads(os.cpu_count())
    cfg = O.base_config(use_vision_tokenizer=True)
    sd = O.make_state_dict(cfg, seed=0)
    train = [v.requires_grad_(True) for k, v in sd.items() if not k.startswith("vqkd.")]
    optim = torch.optim.AdamW(train, lr=1e-4, betas=(0.9, 0.98), eps=1e-8, weight_decay=0.01)
    batch = O.make_batch(cfg, B, L=40, M=15, seed=1, image_uniform=True)
    import random
    import numpy as np
    random.seed(1234)
    np.random.seed(1234)

    def step():
        ids_mask = O.sample_mim_masks(cfg, B)
        ineg = torch.roll(torch.arange(B), 1)
        tneg = torch.roll(torch.arange(B), -1)
        out = O.pretrain_forward(sd, cfg, batch, ineg, tneg, ids_mask=ids_mask)
        loss = out["loss_itc"] + out["loss_itm"] + out["loss_mlm"] + out["loss_mim"]
        optim.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(train, 1.0)
        optim.step()
        return float(loss.detach())
    return step


def cpu_baseline(args, quick):
    B = 2
    step = _oracle_step_fn(B)
    step()
    n = 2 if quick else args.steps
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    dt = (time.perf_counter() - t0) / n
    return {"value": B / dt, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "s_per_step": dt,
            "sample": f"{n} fwd+bwd+AdamW steps of the same workload at {B} pairs/step (oracle/xfm_oracle.py, fp32, eval-mode "
                      f"dropout), after 1 warm-up step"}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    B = 2   # same pairs/step as the cpu_baseline leg of the GPU arm (ITC / ITM are degenerate at one pair)
    step = _oracle_step_fn(B)
    for _ in range(max(1, args.warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    v = B / dt
    sample = (f"each step = fwd+bwd+clip+AdamW of the same workload on {B} pairs (oracle port of the reference algorithm, fp32, "
              f"{os.cpu_count()} host threads)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "XFM-base pretraining step ITC+ITM+MLM+MIM(VQ-KD), 224px / 40 tokens / 15 masked, "
                               "fwd+bwd+clip+AdamW", "pairs_per_step": B, "parallelism": "cpu"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU (pre-train yaml: 96; fine-tune configs: 32 / 64 / 24)")
    ap.add_argument("--config", default="pretrain", choices=["pretrain", "retrieval", "nlvr", "vqa"],
                    help="pretrain = BASELINE configs[1] (the headline); retrieval / nlvr / vqa = configs[2..4] at --res")
    ap.add_argument("--res", type=int, default=384, help="image resolution of the fine-tune configs")
    ap.add_argument("--graph", dest="graph", action="store_true", default=True,
                    help="pretrain config: time the step replayed as one CUDA graph and report it as the headline (default)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="headline = the launch-by-launch sequence")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-eager", action="store_true", help="skip the gpu_eager_baseline leg (eager PyTorch on the same GPU)")
    ap.add_argument("--overlap", default="auto", help="accelerator OVERLAP_ALLREDUCE: auto | true | false")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="pretrain config: write what the last step of the headline timed loop returned (loss, its four "
                         "terms, gradient norm, a seeded sample of the updated fp32 weights) as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != "pretrain"):
        ap.error("--dump-outputs is implemented for the pre-training step (--impl ours --config pretrain)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.overlap = {"true": True, "false": False}.get(str(args.overlap).lower(), "auto")
    args.batch_given = args.batch is not None
    if args.batch is None:
        args.batch = int(os.environ.get("XFM_BENCH_PAIRS", "96"))
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "pretrain":
        if int(os.environ.get("RANK", "0")) == 0:
            run_finetune(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
