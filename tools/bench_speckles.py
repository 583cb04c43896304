"""Speckle removal (bicos_b200_filter_speckles) on the disparities of bench.py's workload and on adversarial scenes.

Disparities, 2048 x 1536: float32 subpixel from a real match of bench.py's 2 x 33 uint8 stacks (LIMITED, thr 0.96,
min_var 2.0, subpixel 0.1, Consistency{1}, bench.py's configuration; speckles set to NaN) and int16 from the same
stacks without a threshold (speckles set to -32768), each filtered with max_diff 1 and max_speckle_size 100 and 1000;
and three adversarial float32 scenes with max_diff 0 and max_speckle_size 100: a one-pixel-wide serpentine through
the whole frame (one component, long union chains across tiles), one component covering the frame (every tile root
joins one root) and a checkerboard of singletons (every pixel a speckle). Reports, as medians over interleaved
rounds in one process:
  us             one call (four launches) between CUDA events, on a fresh copy of the disparity made just before
                 (the copy is outside the events; the 12.6 MB disparity and the 25 MB of labels stay in the 126 MB L2)
  kernel_us      device time of each of the four kernels, from torch.profiler in a separate pass
  pixels, speckles   what the filter removed
  bytes          what the four passes must move: the disparity read twice, the 8 B of labels per pixel written once
                 and read once more (4 B in the flatten pass, 4 B in the write pass), and the pixels set written;
                 hbm_fraction = bytes / time / 7.7 TB/s (HGX B200 data sheet, one GPU)
  match_ms       bench.py's match alone, for scale
  cv2_ms         cv2.filterSpeckles of the int16 frame on one host core of the same machine, where cv2 is installed

    python tools/bench_speckles.py [--rounds 7] [--steps 20] [--out FILE]
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import libbicos_b200 as lb  # noqa: E402
from libbicos_b200 import synth  # noqa: E402

N_IMAGES, ROWS, COLS = 33, 1536, 2048
CFG = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
MARKER = -32768


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return f"{name} ({q})"


def scenes():
    r, c = np.mgrid[0:ROWS, 0:COLS]
    serp = np.full((ROWS, COLS), np.nan, np.float32)
    serp[0::2, :] = 100
    for y in range(1, ROWS, 2):
        serp[y, COLS - 1 if (y // 2) % 2 == 0 else 0] = 100
    return {"serpentine": serp, "covering": np.full((ROWS, COLS), 42, np.float32),
            "checkerboard": np.where((r + c) % 2 == 0, 10, 30).astype(np.float32)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20, help="measurements per case and round")
    ap.add_argument("--out", help="also write the JSON lines here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    h = lb.Handle(0)
    frame = synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, frame=0, xp=torch, device="cuda")[:2]
    cfg_f, cfg_i = lb.Config(**CFG), lb.Config(nxcorr_threshold=None)
    sub, _ = h.match(*frame, cfg_f)
    i16, _ = h.match(*frame, cfg_i)
    torch.cuda.synchronize()
    # (name, pristine disparity, new_value, max_speckle_size, max_diff)
    cases = [(f"float32 subpixel, size {s}", sub, float("nan"), s, 1.0) for s in (100, 1000)]
    cases += [(f"int16, size {s}", i16, MARKER, s, 1.0) for s in (100, 1000)]
    cases += [(f"{k} (float32)", torch.from_numpy(v).cuda(), MARKER, 100, 0.0) for k, v in scenes().items()]
    work = {name: src.clone() for name, src, *_ in cases}

    counts = {}
    for name, src, nv, size, diff in cases:  # warm-up, and what each case removes
        work[name].copy_(src)
        _, c = h.filter_speckles(work[name], nv, size, diff, counts=True)
        counts[name] = c
    ms = {name: [] for name, *_ in cases}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for name, src, nv, size, diff in cases:
            for _ in range(args.steps):
                work[name].copy_(src)
                e0.record()
                h.filter_speckles(work[name], nv, size, diff)
                e1.record()
                e1.synchronize()
                ms[name].append(e0.elapsed_time(e1))
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    match_ms = []
    for _ in range(args.steps):
        m0.record()
        h.match(*frame, cfg_f)
        m1.record()
        m1.synchronize()
        match_ms.append(m0.elapsed_time(m1))

    # device time of each kernel, in a pass of its own under the profiler
    from torch.profiler import ProfilerActivity, profile

    kernel_us = {}
    for name, src, nv, size, diff in cases:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                work[name].copy_(src)
                h.filter_speckles(work[name], nv, size, diff)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            for k in ("tile", "border", "flatten", "write"):
                if f"speckle_{k}_kernel" in ev.name:
                    per.setdefault(k, []).append(getattr(ev, "device_time_total", None) or ev.cuda_time_total)
        kernel_us[name] = {k: round(float(np.median(v)), 2) for k, v in per.items()}

    cv2_ms = None
    try:
        import cv2

        host = i16.cpu().numpy()
        t = []
        for _ in range(5):
            a = host.copy()
            t0 = time.perf_counter()
            cv2.filterSpeckles(a, MARKER, 100, 1)
            t.append((time.perf_counter() - t0) * 1e3)
        cv2_ms = round(float(np.median(t)), 2)
    except ImportError:
        pass

    gpu = gpu_info()
    px = ROWS * COLS
    lines = []
    for name, src, nv, size, diff in cases:
        eb = src.element_size()
        med = float(np.median(ms[name]))
        nbytes = 2 * px * eb + px * 8 + px * 8 + counts[name]["pixels"] * eb
        lines.append(json.dumps(dict(
            workload=f"filter_speckles 2048x1536 {name}, max_diff {diff}", gpu=gpu, new_value=str(nv), max_speckle_size=size,
            pixels=counts[name]["pixels"], speckles=counts[name]["speckles"], us=round(med * 1e3, 2),
            us_spread=[round(min(ms[name]) * 1e3, 2), round(max(ms[name]) * 1e3, 2)], kernel_us=kernel_us[name], bytes=nbytes,
            hbm_fraction=round(nbytes / (med * 1e-3) / HBM_BYTES_PER_S, 3), target_us=50.0,
            match_ms=round(float(np.median(match_ms)), 4), share_of_match=round(med / float(np.median(match_ms)), 4),
            cv2_ms=cv2_ms if name.startswith("int16, size 100") else None, rounds=args.rounds, steps=args.steps)))
        print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
