"""Reprojection stage (bicos_b200_reproject) on the disparity of bench.py's workload.

Disparities: 2048 x 1536 from real matches of bench.py's 2 x 33 uint8 stacks, float32 subpixel (LIMITED, thr 0.96,
min_var 2.0, subpixel 0.1, Consistency{1}, bench.py's configuration) and int16 (the same stacks without a threshold).
Q is shaped like cv2.stereoRectify's output (f = 1400 px, baseline 0.12, principal points 3.5 px apart). Reports,
as medians over interleaved rounds in one process:
  hot_us[mode]    one call right after the match that wrote its disparity (disparity in L2): CUDA events from the
                  end of the match to the end of the call, for mode = dense (xyz only), points (list + index +
                  counts) and both
  cold_us[mode]   one call while cycling over COLD_FRAMES disparity copies with their own outputs (about 400 MB,
                  beyond the 126 MB L2), events around all of them after a match (the calls are enqueued while the
                  match runs, so host launch time is not measured)
  bytes[mode]     what the call must move: every disparity pixel read once, 12 B per pixel for dense, 16 B per kept
                  point for the list; hbm_fraction = bytes / cold time / 7.7 TB/s (HGX B200 data sheet, one GPU)
  match_ms / match_reproject_ms   a match alone against a match followed by reproject(both) of its disparity
  kernel_us       device time of reproject_kernel itself per mode, from torch.profiler in a separate pass

    python tools/bench_reproject.py [--rounds 7] [--steps 20] [--out FILE]
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import libbicos_b200 as lb  # noqa: E402
from libbicos_b200 import synth  # noqa: E402

N_IMAGES, ROWS, COLS, COLD_FRAMES = 33, 1536, 2048, 4
CFG = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
MODES = ("dense", "points", "both")


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return f"{name} ({q})"


def stereo_q():
    cx, cy, f, tx, dcx = (COLS - 1) / 2.0, (ROWS - 1) / 2.0, 1400.0, -0.12, 3.5
    return np.array([[1, 0, 0, -cx], [0, 1, 0, -cy], [0, 0, 0, f], [0, 0, -1.0 / tx, dcx / tx]])


class Slot:
    """A disparity with its own output buffers, called through the C ABI without host work beyond the launch."""

    def __init__(self, h, disp, q):
        self.h, self.disp, self.q = h, disp, q
        self.code = lb.capi.TYPE_16S if disp.dtype == torch.int16 else lb.capi.TYPE_32F
        self.xyz = torch.empty((ROWS, COLS, 3), dtype=torch.float32, device="cuda")
        self.points = torch.empty((ROWS * COLS, 3), dtype=torch.float32, device="cuda")
        self.index = torch.empty((ROWS * COLS,), dtype=torch.int32, device="cuda")
        self.counts = torch.empty((4,), dtype=torch.int64, device="cuda")

    def __call__(self, mode):
        dense = mode in ("dense", "both")
        pts = mode in ("points", "both")
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        rc = lb.lib().bicos_b200_reproject(self.h._h, self.disp.data_ptr(), self.code, self.disp.stride(0) * self.disp.element_size(),
                                           ROWS, COLS, self.q, 0, self.xyz.data_ptr() if dense else None, COLS * 12,
                                           self.points.data_ptr() if pts else None, self.index.data_ptr() if pts else None,
                                           self.counts.data_ptr() if pts else None, st)
        if rc != 0:
            raise lb.BicosError(lb.lib().bicos_b200_last_error().decode())


def after_match(h, frame, cfg, out, calls):
    """Device ms of `calls` enqueued behind a match: from the match's end to the last call's end."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h.match(*frame, cfg, out=out)
    e0.record()
    for c in calls:
        c()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20, help="measurements per quantity and round")
    ap.add_argument("--out", help="also write the JSON lines here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")

    h = lb.Handle(0)
    q = h._q_matrix(stereo_q())
    frames = [synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, frame=f, xp=torch, device="cuda")[:2] for f in range(2)]
    lines = []
    for label, cfg in (("float32 subpixel", lb.Config(**CFG)), ("int16", lb.Config(nxcorr_threshold=None))):
        outs = [h.match(*fr, cfg) for fr in frames]
        torch.cuda.synchronize()
        hot = [Slot(h, o[0], q) for o in outs]
        cold = [Slot(h, outs[k % 2][0].clone(), q) for k in range(COLD_FRAMES)]
        for s in hot + cold:
            for m in MODES:
                s(m)
        torch.cuda.synchronize()
        counts = [int(v) for v in hot[0].counts.cpu()]
        kept = counts[0]
        ms = {f"hot_{m}": [] for m in MODES}
        ms.update({f"cold_{m}": [] for m in MODES})
        ms.update(match=[], match_reproject=[])
        for _ in range(args.rounds):
            for m in MODES:
                for k in range(args.steps):
                    f = k % 2
                    ms[f"hot_{m}"].append(after_match(h, frames[f], cfg, outs[f], [lambda s=hot[f], m=m: s(m)]))
                    ms[f"cold_{m}"].append(after_match(h, frames[f], cfg, outs[f], [lambda s=s, m=m: s(m) for s in cold])
                                           / COLD_FRAMES)
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            for k in range(args.steps):
                f = k % 2
                e[0].record()
                h.match(*frames[f], cfg, out=outs[f])
                e[1].record()
                e[2].record()
                h.match(*frames[f], cfg, out=outs[f])
                hot[f]("both")
                e[3].record()
                e[3].synchronize()
                ms["match"].append(e[0].elapsed_time(e[1]))
                ms["match_reproject"].append(e[2].elapsed_time(e[3]))
        med = {k: float(np.median(v)) for k, v in ms.items()}

        # kernel device time alone, in a pass of its own under the profiler
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for m in MODES:
                for _ in range(10):
                    for s in cold:
                        s(m)
                torch.cuda.synchronize()
        kern = {}
        tags = {"both": (", true, true>", "Lb1ELb1E"), "dense": (", true, false>", "Lb1ELb0E"), "points": (", false, true>", "Lb0ELb1E")}
        for ev in prof.events():
            if "reproject_kernel" in ev.name:
                mode = next((m for m, t in tags.items() if any(x in ev.name for x in t)), ev.name)
                kern.setdefault(mode, []).append(getattr(ev, "device_time_total", None) or ev.cuda_time_total)
        kernel_us = {m: round(float(np.median(v)), 2) for m, v in kern.items()}

        px = ROWS * COLS
        eb = 2 if label == "int16" else 4
        nbytes = {"dense": px * (eb + 12), "points": px * eb + kept * 16, "both": px * (eb + 12) + kept * 16}
        line = dict(workload=f"reproject 2048x1536 {label} disparity of bench.py's stacks ({CFG if label != 'int16' else 'no threshold'}), "
                             f"stereoRectify-shaped Q", gpu=gpu_info(), kept=kept, invalid=counts[1], non_finite=counts[2],
                    negative_z=counts[3],
                    hot_us={m: round(med[f"hot_{m}"] * 1e3, 2) for m in MODES},
                    cold_us={m: round(med[f"cold_{m}"] * 1e3, 2) for m in MODES},
                    cold_us_spread={m: [round(min(ms[f"cold_{m}"]) * 1e3, 2), round(max(ms[f"cold_{m}"]) * 1e3, 2)] for m in MODES},
                    kernel_us=kernel_us, bytes=nbytes,
                    hbm_fraction={m: round(nbytes[m] / (med[f"cold_{m}"] * 1e-3) / HBM_BYTES_PER_S, 3) for m in MODES},
                    target_us_both=30.0, match_ms=round(med["match"], 4), match_reproject_ms=round(med["match_reproject"], 4),
                    reproject_share_of_match=round((med["match_reproject"] - med["match"]) / med["match"], 4),
                    rounds=args.rounds, steps=args.steps)
        lines.append(json.dumps(line))
        print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
