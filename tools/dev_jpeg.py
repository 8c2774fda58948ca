"""Baseline JPEG decode on the GPU (feed.decode_jpeg, csrc/jpeg.cu) against Pillow on the host.

Input: seeded synthetic 640 x 480, quality-90, 4:2:0 JPEGs in batches of 96 and 1024, and the same images with a restart
marker every MCU row (DRI).  Per batch: device time of each of the three decode kernels (torch.profiler CUDA
kernel times after a synchronise, warmed up, median of --reps), end to end from host bytes to decoded device buffer (host clock around
decode_jpeg, which ends with its status read), and Pillow `Image.open(f).convert("RGB")` of the same bytes on 1 and N threads.
Card name and power limit are read in the same run.  One JSON line per measurement on stdout and in --out."""
import argparse
import io
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from xfm_b200 import feed, lib  # noqa: E402


def make_batch(n, dri, seed=0):
    from PIL import Image
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:480, 0:640]
    out = []
    for i in range(n):
        base = np.stack([(xx * (1 + i % 3) + yy) % 256, (yy * 2 + i) % 256, (xx + 3 * yy) % 256], -1)
        img = np.clip(base + rng.normal(0, 12, base.shape), 0, 255).astype(np.uint8)
        f = io.BytesIO()
        Image.fromarray(img).save(f, "JPEG", quality=90, subsampling=2, **({"restart_marker_rows": 1} if dri else {}))
        out.append(f.getvalue())
    return out


def stage_times(blobs, reps):
    """Median per-kernel device time (ms) of the three decode launches, timed one launch at a time."""
    info = lib.jpeg_plan(blobs)
    assert (info[:, 0] == 0).all()
    B = len(blobs)
    offs = np.zeros((B, 4), np.int64)
    for col, size in ((0, np.array([len(b) for b in blobs])), (1, info[:, 4]), (2, info[:, 5]), (3, info[:, 1] * info[:, 2] * 3)):
        offs[:, col] = np.cumsum(size) - size
    desc, iv = lib.jpeg_tables(blobs, info, offs)
    dev = dict(device="cuda")
    data = torch.frombuffer(bytearray(b"".join(blobs)), dtype=torch.uint8).cuda()
    desc, iv = desc.cuda(), iv.cuda()
    coef = torch.empty((int(info[:, 4].sum()), 64), dtype=torch.int16, **dev)
    planes = torch.empty(int(info[:, 5].sum()), dtype=torch.uint8, **dev)
    out = torch.empty(int((info[:, 1] * info[:, 2] * 3).sum()), dtype=torch.uint8, **dev)
    status = torch.zeros(B, dtype=torch.int32, **dev)
    args = (data, desc, iv, B, coef, planes, out, status, int(info[:, 4].max()), int(info[:, 1].max()), int(info[:, 2].max()))
    for _ in range(3):
        lib.jpeg_decode(*args)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            lib.jpeg_decode(*args)
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "jpeg_" in e.name:
            per.setdefault(e.name.split("(")[0].replace("xfm::", ""), []).append(e.device_time_total / 1000.0)
    assert int(status.sum()) == 0
    return {k: float(np.median(v)) for k, v in per.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="96,1024")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "dev_jpeg.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dev_jpeg.py measures the GPU decoder: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()
    rows = []
    for n in [int(v) for v in a.batches.split(",")]:
        for dri in (False, True):
            blobs = make_batch(n, dri)
            ref = feed._pil_rgb(blobs[0]).numpy()
            stages = stage_times(blobs, a.reps)
            for _ in range(2):
                feed.decode_jpeg(blobs)
            torch.cuda.synchronize()
            e2e = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                out, meta, nfb = feed.decode_jpeg(blobs)
                e2e.append((time.perf_counter() - t0) * 1e3)
            assert nfb == 0 and np.array_equal(out[:640 * 480 * 3].view(480, 640, 3).cpu().numpy(), ref)
            t0 = time.perf_counter()
            for b in blobs[:min(n, 96)]:
                feed._pil_rgb(b)
            pil1 = (time.perf_counter() - t0) * 1e3 / min(n, 96) * n
            with ThreadPoolExecutor(a.threads) as ex:
                list(ex.map(feed._pil_rgb, blobs[:8]))
                t0 = time.perf_counter()
                list(ex.map(feed._pil_rgb, blobs))
                pilN = (time.perf_counter() - t0) * 1e3
            row = dict(card=card, batch=n, dri=dri, bytes_per_image=float(np.mean([len(b) for b in blobs])),
                       stage_ms=stages, device_ms=sum(stages.values()), end_to_end_ms=float(np.median(e2e)),
                       pillow_1thread_ms=pil1, pillow_threads=a.threads, pillow_nthread_ms=pilN)
            print(json.dumps(row), flush=True)
            rows.append(row)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
