"""Rectification stage (bicos_b200_remap) and match_rectified against match, on bench.py's workload.

2 x 33 uint8 2048 x 1536 stacks of the synthetic scene (LIMITED, thr 0.96, min_var 2.0, subpixel 0.1, Consistency{1}),
treated as raw camera images, and float32 maps of the same size from synth.rectify_maps: a pinhole camera with radial
distortion (k1 = -0.12, k2 = 0.03) and a small rotation, mirrored between the two cameras, i.e. what
cv2.initUndistortRectifyMap produces for such a rig. Reports, as medians over interleaved rounds in one process:
  remap_ms       both stacks through Handle.remap (two stage launches), CUDA events around back-to-back pairs
  match_ms / match_rectified_ms   a frame through Handle.match on rectified stacks / Handle.match_rectified on raw ones
  hbm_*          the bytes the remap must move (every source and output pixel once, both maps) over remap_ms, and the
                 share of the B200's 7.7 TB/s data-sheet HBM bandwidth that rate is
  cv2_ms_per_stack   cv2.remap of the 33 planes of one stack on the host, only when cv2 is importable
Frames alternate between FRAMES stereo pairs, so the working set (about 470 MB per frame for the remap) exceeds the
126 MB L2.

    python tools/bench_rectify.py [--rounds 5] [--steps 10] [--out FILE]
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

N_IMAGES, ROWS, COLS, FRAMES = 33, 1536, 2048, 2
CFG = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return f"{name} ({q})"


def timed(fn, steps):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()  # warm-up
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    ev1.synchronize()
    return ev0.elapsed_time(ev1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10, help="passes over the frames per measurement and round")
    ap.add_argument("--out", help="also write the JSON lines here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    h = lb.Handle(0)
    frames = [synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, frame=f, xp=torch, device="cuda")[:2] for f in range(FRAMES)]
    host_maps = [synth.rectify_maps(ROWS, COLS, camera=c) for c in (0, 1)]
    maps = lb.RectifyMaps(*[torch.from_numpy(m).cuda() for pair in host_maps for m in pair])
    cfg = lb.Config(**CFG)
    rect = [(h.remap(l, maps.map_x0, maps.map_y0), h.remap(r, maps.map_x1, maps.map_y1)) for l, r in frames]
    outs = [h.match(*rl, cfg) for rl in rect]
    outs_r = [h.match_rectified(l, r, maps, cfg) for l, r in frames]
    torch.cuda.synchronize()
    same = all(torch.equal(a[0].nan_to_num(7.0), b[0].nan_to_num(7.0)) and torch.equal(a[1].nan_to_num(7.0), b[1].nan_to_num(7.0))
               for a, b in zip(outs, outs_r))

    def remap_pass():
        for (l, r), (rl, rr) in zip(frames, rect):
            h.remap(l, maps.map_x0, maps.map_y0, out=rl)
            h.remap(r, maps.map_x1, maps.map_y1, out=rr)

    def match_pass():
        for rl, out in zip(rect, outs):
            h.match(*rl, cfg, out=out)

    def rectified_pass():
        for (l, r), out in zip(frames, outs_r):
            h.match_rectified(l, r, maps, cfg, out=out)

    ms = {"remap": [], "match": [], "match_rectified": []}
    for _ in range(args.rounds):
        ms["remap"].append(timed(remap_pass, args.steps) / FRAMES)
        ms["match"].append(timed(match_pass, args.steps) / FRAMES)
        ms["match_rectified"].append(timed(rectified_pass, args.steps) / FRAMES)
    med = {k: float(np.median(v)) for k, v in ms.items()}

    px = ROWS * COLS
    remap_bytes = 2 * (2 * N_IMAGES * px + 2 * 4 * px)  # per side: every source and output pixel once, two float32 maps
    rate = remap_bytes / (med["remap"] * 1e-3)
    line = dict(workload=f"2x{N_IMAGES} uint8 {COLS}x{ROWS}, maps {COLS}x{ROWS} float32, {CFG}", gpu=gpu_info(),
                remap_ms=round(med["remap"], 4), remap_ms_spread=[round(min(ms["remap"]), 4), round(max(ms["remap"]), 4)],
                remap_target_ms=0.15, remap_bytes=remap_bytes, hbm_tb_per_s=round(rate / 1e12, 3),
                hbm_fraction=round(rate / HBM_BYTES_PER_S, 3), match_ms=round(med["match"], 4),
                match_rectified_ms=round(med["match_rectified"], 4),
                rectify_overhead_ms=round(med["match_rectified"] - med["match"], 4),
                match_rectified_equals_match_of_remap=bool(same), rounds=args.rounds, frames_per_round=args.steps * FRAMES)
    try:
        import cv2

        left = frames[0][0].cpu().numpy()
        mx, my = host_maps[0]
        cv2.remap(left[0], mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        t0 = time.perf_counter()
        for t in range(N_IMAGES):
            cv2.remap(left[t], mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        line["cv2_ms_per_stack"] = round((time.perf_counter() - t0) * 1e3, 2)
        line["cv2_threads"] = cv2.getNumThreads()
        line["cv2_host_cpus"] = os.cpu_count()
    except ImportError:
        line["cv2_ms_per_stack"] = None
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
