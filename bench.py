#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200: Mpx/s of disparity output.

Workload (BASELINE.json `metric` + configs[1]'s Config): 2 x 33-image uint8 2048x1536 stacks,
LIMITED transform, nxcorr_threshold 0.96, min_variance 2.0, subpixel_step 0.1,
Variant::Consistency{max_lr_diff=1}, float precision.

One step = one pass of BICOS::match over a batch of FRAMES distinct synthetic stereo stacks per
GPU (frame-sharded across GPUs, weak scaling, no data-path collective: frames are independent).
  value      whole-job Mpx/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e        same metric through the host-buffer C-ABI entry point (bicos_b200_match_host, what
             pybicos' BICOS_Match calls): pinned host stacks in, host disparity + corrmap out,
             copies inside the timed region
  roofline   the dominant kernel (row-wise Hamming search). Tensor-core engine (default): int8 TOP/s
             against the dense int8 rate measured live with cuBLASLt; the popcount engine is timed on the
             same frames and reported as roofline.other_engine: algorithmic popc32/s against the
             measured pure-POPC issue rate of this GPU; the two HBM-bound kernels are listed
             under roofline_other against MEASURED_PEAKS.json
  cpu_baseline  the unmodified reference CPU backend (oracle/_ref) on a bounded row sample

`--impl reference` times the reference's own CPU implementation on the host cores instead.

`--dump-outputs DIR` writes what the timed path returned in its last step, so that two builds can be compared
output for output: disparity_<f>.npy and corrmap_<f>.npy (float32, [DUMP_ROWS, 2048]) for every frame f of
rank 0, on the same rows of every frame, drawn once with a fixed seed. The library marks invalid disparities
and corrmap cells it never evaluated as NaN; the dump keeps every value finite: such cells are written as 0 and
disparity_valid_<f>.npy / corrmap_valid_<f>.npy (float32, 1 = a number, 0 = NaN) say which they are (48 MiB in
all). The frames are a pure function of their index (libbicos_b200/synth.py), so the same arguments give the
same inputs in every run.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line. Libraries write to file descriptor 1 behind Python's back (NCCL prints
# its version banner there at every level from VERSION up, WARN included): Python's sys.stdout keeps a duplicate
# of the original descriptor, and descriptor 1 itself is pointed at stderr for everything else.
sys.stdout.flush()
sys.stdout = os.fdopen(os.dup(1), "w", buffering=1)
os.dup2(2, 1)

N_IMAGES, ROWS, COLS = 33, 1536, 2048
FRAMES = 4  # distinct stereo stacks per GPU per step (4 x 208 MB of input > 126 MB L2)
CFG = dict(nxcorr_threshold=0.96, min_variance=2.0, subpixel_step=0.1, consistency=True, max_lr_diff=1)
WORKLOAD = ("2x33 uint8 2048x1536, LIMITED, thr 0.96, min_var 2.0, subpixel_step 0.1, "
            "Consistency{max_lr_diff=1}, float")
# one dictionary for both arms (the driver compares them): what is specific to an arm says so in its value
CONFIG = {
    "workload": WORKLOAD,
    "frames_per_gpu_per_step": FRAMES,
    "sharding": "frame-sharded, one process per GPU, no data-path collective; the frames of a step are one bicos_b200_match_batch",
    "l2": f"inputs larger than L2 ({FRAMES} x 208 MB per GPU per step); no explicit flush",
    "reference_arm_sample": "a bounded row sample of one stereo stack per step (cost is linear in rows), see cpu_baseline.sample",
}
DUMP_ROWS, DUMP_SEED = 384, 20261020


def dump_outputs(directory, outs):
    """--dump-outputs: the (disparity, corrmap) pairs of one step, on a fixed seeded sample of rows; NaN cells as 0
    beside a float validity mask, so that every value written is finite."""
    import numpy as np
    import torch

    os.makedirs(directory, exist_ok=True)
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(ROWS, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(outs[0][0].device)
    for f, (disp, corr) in enumerate(outs):
        for name, a in (("disparity", disp), ("corrmap", corr)):
            a = a.index_select(0, idx)
            valid = torch.isfinite(a)
            np.save(os.path.join(directory, f"{name}_{f}.npy"), torch.where(valid, a, torch.zeros_like(a)).cpu().numpy())
            np.save(os.path.join(directory, f"{name}_valid_{f}.npy"), valid.to(a.dtype).cpu().numpy())


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(p.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax = float(parts[1])
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_cpus(local):
    """Pin this process to the CPUs next to its GPU (NVML's ideal set) before any pinned host
    buffer is allocated, so that on a multi-socket host the staging buffers of a rank live on its
    GPU's NUMA node (no effect on a single-node host). Returns a short description for the JSON line."""
    try:
        import pynvml
        import torch

        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode() if not uuid.startswith("GPU-") else uuid.encode())
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        return f"nvml ideal cpus ({len(os.sched_getaffinity(0))} cpus)"
    except Exception as e:  # affinity is an optimisation, never a requirement
        return f"unbound ({type(e).__name__})"


def measure_popc_peak(sm_max_mhz):
    """Pure-POPC issue rate of this GPU (tools/microbench, same binary as profiles/microbench_*.txt)."""
    exe = os.path.join(ROOT, "tools", "microbench")
    if os.path.exists(exe):
        try:
            out = subprocess.run([exe, "--popc"], capture_output=True, text=True, timeout=60).stdout
            for line in out.splitlines():
                if line.startswith("POPC_PER_S"):
                    return float(line.split()[1]), "measured (tools/microbench --popc)"
        except Exception:
            pass
    return 16.0 * 148 * sm_max_mhz * 1e6, "nominal 16 POPC/clk/SM x 148 SM x max clock"


def measure_int8_peak():
    """Dense int8 tensor-core rate of this GPU: cuBLASLt through torch._int_mm, 8192^3, best of 10 (TOP/s)."""
    import torch

    try:
        a = torch.randint(-8, 8, (8192, 8192), dtype=torch.int8, device="cuda")
        b = torch.randint(-8, 8, (8192, 8192), dtype=torch.int8, device="cuda").t().contiguous().t()
        torch._int_mm(a, b)
        best = float("inf")
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * 8192**3 / (best * 1e-3) / 1e12, "measured live (torch._int_mm 8192^3 = cuBLASLt int8, best of 10, CUDA events)"
    except Exception as e:  # noqa: BLE001
        bf16 = 1632.7
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                bf16 = float(json.load(f)["bf16_tflops"])
        except (OSError, KeyError, ValueError):
            pass
        return 2 * bf16, f"2 x the measured dense bf16 rate of MEASURED_PEAKS.json (torch._int_mm failed: {type(e).__name__})"


def cpu_reference_run(rows, threads=None, keep=None):
    """Reference CPU backend on `rows` rows of frame 0 of the workload. Returns (seconds, kind, cores).
    `keep` (a dict) receives row0 and the reference's outputs, for the parity check of the bench line."""
    import numpy as np

    import oracle
    from libbicos_b200 import synth

    lib, kind = (oracle.ref, "reference") if oracle.ref.available() else (oracle.port, "port")
    if not lib.available():
        oracle.build(ref=False)
    left, right, _ = synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, row0=ROWS // 2 - rows // 2, rows=rows)
    if threads:
        lib.set_threads(threads)
    cores = threads or lib.hardware_threads()
    t0 = time.perf_counter()
    disp, corr = lib.match(left, right, **CFG)
    t = time.perf_counter() - t0
    if keep is not None:
        keep.update(row0=ROWS // 2 - rows // 2, rows=rows, disp=disp, corr=corr)
    return t, kind, cores


def parity_against_reference(keep, disp, corr, kind):
    """The bench's own frame 0 (GPU, the kernels that were timed) against the reference CPU backend on the same
    rows. north_star tolerances: valid mask bit-exact except where the NXC lies within 1e-6 of the threshold,
    corrmap within 1e-5, subpixel disparity within 1e-3 px."""
    import numpy as np

    r0, rows = keep["row0"], keep["rows"]
    gd, gc = disp[r0 : r0 + rows], corr[r0 : r0 + rows]
    wd, wc = keep["disp"], keep["corr"]
    inv_g, inv_w = np.isnan(gd), np.isnan(wd)
    edge = np.abs(np.nan_to_num(wc, nan=9.0) - CFG["nxcorr_threshold"]) < 1e-6
    mask_mismatch = int(((inv_g != inv_w) & ~edge).sum())
    both = ~(inv_g | inv_w)
    okc = ~np.isnan(wc) & ~np.isnan(gc)
    out = {
        "against": f"oracle/{'_ref (unmodified reference CPU backend)' if kind == 'reference' else 'port'}",
        "frame": 0, "row0": r0, "rows": rows, "pixels": int(gd.size), "valid": int(both.sum()),
        "mask_mismatch": mask_mismatch, "threshold_edge_pixels": int(edge.sum()),
        "corr_nan_mismatch": int((np.isnan(gc) != np.isnan(wc)).sum()),
        "disp_max_abs": float(np.max(np.abs(gd[both] - wd[both]), initial=0.0)),
        "corr_max_abs": float(np.max(np.abs(gc[okc] - wc[okc]), initial=0.0)),
        "bit_identical": bool(np.array_equal(gd, wd, equal_nan=True) and np.array_equal(gc, wc, equal_nan=True)),
    }
    out["within_north_star"] = bool(out["mask_mismatch"] == 0 and out["corr_nan_mismatch"] == 0
                                    and out["disp_max_abs"] <= 1e-3 and out["corr_max_abs"] <= 1e-5)
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = 32
    for _ in range(max(args.warmup, 1)):
        t, kind, cores = cpu_reference_run(rows)
    # size the per-step sample so that the whole run stays within a few minutes
    rows = int(min(ROWS, max(16, rows * (8.0 / max(t, 1e-3)))))
    times = []
    for _ in range(args.steps):
        t, kind, cores = cpu_reference_run(rows)
        times.append(t)
    ms = 1e3 * sum(times) / len(times)
    value = rows * COLS / (ms * 1e-3) / 1e6
    sample = f"{rows} of {ROWS} rows of one 2048-wide stereo stack per step (cost is linear in rows)"
    line = {
        "impl": "reference", "metric": "Mpx/s disparity", "value": value, "unit": "Mpx/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": CONFIG,
        "cpu_baseline": {"value": value, "unit": "Mpx/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--table", action="store_true",
                    help="instead of the bench line: every BASELINE config (tools/bench_configs.py) with the "
                         "reference's CUDA backend timed beside it, one JSON line per config")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the disparity and corrmap of the last step's frames to "
                         "DIR/<name>.npy (float32, a fixed seeded sample of rows; NaN cells as 0 beside validity masks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.table):
        ap.error("--dump-outputs dumps the timed path of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.table:
        import oracle  # baselines are timed beside the product, never inside it
        from tools import bench_configs

        bench_configs.run_table(["C1", "C2", "metric", "C3", "C3n20", "C4", "C5"], 10,
                                oracle.refcuda if oracle.refcuda.available() else None)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import libbicos_b200 as lb
    from libbicos_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # fewer ranks than visible GPUs: spread them over the node's PCIe tree (the end-to-end path is bound by the
    # host link, which neighbouring GPUs share); BICOS_BENCH_DEVICES=first keeps LOCAL_RANK = ordinal
    from libbicos_b200 import topology

    if os.environ.get("BICOS_BENCH_DEVICES", "") == "first":
        devices, device_policy = list(range(world)), "LOCAL_RANK = ordinal (BICOS_BENCH_DEVICES=first)"
    else:
        devices, device_policy = topology.pick_devices(world)
    local = devices[local_rank]
    torch.cuda.set_device(local)
    all_cpus = os.sched_getaffinity(0)
    affinity = bind_to_gpu_cpus(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    hbm_peak, hbm_src, sm_max = load_peaks()
    cfg = lb.Config(**CFG)
    h = lb.Handle(local)
    px = ROWS * COLS
    K = lb.descriptor_words(N_IMAGES, False)

    # distinct frames per rank: frame index = rank * FRAMES + f
    frames = [synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, frame=rank * FRAMES + f, xp=torch, device="cuda")[:2]
              for f in range(FRAMES)]
    outs = [h.match(l, r, cfg) for (l, r) in frames]
    torch.cuda.synchronize()

    def step():
        # throughput mode: the FRAMES stereo stacks of a step as one batch (bicos_b200_match_batch: frame f + 1's
        # transform + search beside frame f's refine; the current stream is joined before and after)
        h.match_batch(frames, cfg, outs=outs)

    def step_serial():
        for (l, r), out in zip(frames, outs):
            h.match(l, r, cfg, out=out)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    h.set_profiling(True)
    launches0 = h.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    total_ms = max_over_ranks(ev0.elapsed_time(ev1))
    stage_ms, n_matches = h.stage_times()
    h.set_profiling(False)
    search_kernel = lb.last_search_kernel()  # what the timed matches dispatched, e.g. mma2<K=4,nodupes=0,ct=1,dirs=2>
    launches = h.kernel_launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    # frame 0 as the timed region left it (the engine comparison further down writes into `outs` again)
    timed_frame0 = (outs[0][0].cpu().numpy(), outs[0][1].cpu().numpy()) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)
    ms_per_step = total_ms / args.steps
    value = world * FRAMES * px / (ms_per_step * 1e-3) / 1e6

    # ---- end to end through the host-buffer C-ABI entry point --------------------------------
    host = [(l.cpu().pin_memory().numpy(), r.cpu().pin_memory().numpy()) for (l, r) in frames]
    host_out = [(torch.empty((ROWS, COLS), dtype=torch.float32).pin_memory().numpy(),
                 torch.empty((ROWS, COLS), dtype=torch.float32).pin_memory().numpy()) for _ in frames]

    # two handles = two frames in flight: frame f+1 uploads while frame f is matched and frame
    # f-1 downloads (bicos_b200_match_host_begin / _end); every result is complete in host
    # memory when its step ends
    inflight = max(1, min(int(os.environ.get("BICOS_BENCH_INFLIGHT", "2")), FRAMES))
    hh = [h] + [lb.Handle(local) for _ in range(inflight - 1)]

    def e2e_step():
        for f, ((l, r), out) in enumerate(zip(host, host_out)):
            hh[f % inflight].match_host_end()  # the frame this handle carried in the previous round
            hh[f % inflight].match_host_begin(l, r, cfg, out=out)
        for x in hh:
            x.match_host_end()

    for _ in range(2):
        e2e_step()
    barrier()
    e2e_steps = max(3, args.steps // 2)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    barrier()
    e2e_value = world * FRAMES * px / (e2e_ms * 1e-3) / 1e6
    same = bool(np.array_equal(host_out[0][0], outs[0][0].cpu().numpy(), equal_nan=True))

    # the ceiling of that path: what plain pinned host-to-device copies reach on the same GPUs at the same time
    # (256 MB each, all ranks concurrently; one GPU alone gets about 55 GB/s, GPUs behind one host bridge share it)
    link_host = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    link_dev = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(2):
        link_dev.copy_(link_host, non_blocking=True)
    barrier()
    ev0.record()
    for _ in range(8):
        link_dev.copy_(link_host, non_blocking=True)
    ev1.record()
    barrier()
    link_gbs = 8 * (256 << 20) / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
    if world > 1:
        t = torch.tensor([link_gbs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        link_gbs = float(t.item())
    del link_host, link_dev
    e2e_h2d_gbs = world * FRAMES * 2 * N_IMAGES * px / (e2e_ms * 1e-3) / 1e9

    # ---- N > 1: ONE match of the same workload row-sharded over the N GPUs (strong scaling; BASELINE.json
    #      configs[2] / [3] ask for this mode). Rank g holds rows [g H / N, (g + 1) H / N) of frame 0 and runs the
    #      whole path on them; the refine kernels store their rows into rank 0's images over NVLink peer memory
    #      (sharding.PeerAssembly), so the only exchange is that store. Device time = max over ranks. ----
    row_sharded = None
    if world > 1:
        from libbicos_b200 import sharding

        lo, hi = sharding.row_range(rank, world, ROWS)
        sl, sr = synth.make_stacks(N_IMAGES, ROWS, COLS, np.uint8, row0=lo, rows=hi - lo, xp=torch, device="cuda")[:2]
        pa = sharding.PeerAssembly(h, ROWS, COLS, cfg, local)
        for _ in range(3):
            pa.match(sl, sr)
            pa.finish()
        ts = []
        for _ in range(20):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            pa.match(sl, sr)
            b.record()
            pd, pc = pa.finish()
            ts.append(max_over_ranks(a.elapsed_time(b)))
        shard_kernel = lb.last_search_kernel()
        if rank == 0:
            single = []
            l0, r0 = frames[0]
            for _ in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                h.match(l0, r0, cfg, out=outs[0])
                b.record()
                torch.cuda.synchronize()
                single.append(a.elapsed_time(b))
            single_ms, shard_ms = float(np.median(single)), float(np.median(ts))
            eq = bool(torch.equal(torch.nan_to_num(pd, nan=-7.0), torch.nan_to_num(outs[0][0], nan=-7.0))
                      and torch.equal(torch.nan_to_num(pc, nan=-7.0), torch.nan_to_num(outs[0][1], nan=-7.0)))
            row_sharded = {"ms_per_match": shard_ms, "ms_per_match_min": float(np.min(ts)), "mpx_per_s": px / shard_ms / 1e3,
                           "single_gpu_ms_per_match": single_ms, "speedup_vs_1gpu": single_ms / shard_ms,
                           "rows_per_gpu": hi - lo, "assembly": "peer", "search_kernel_per_shard": shard_kernel,
                           "equals_single_gpu": eq, "scaling": "strong"}
        pa.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ------------------------------------------------------
    popc_peak, popc_src = measure_popc_peak(sm_max)
    t_tr, t_se, t_re = (1e-3 * v / max(n_matches, 1) for v in stage_ms)
    popc_alg = COLS * px * K  # SURVEY 8d: S = W * P * K popc32 per match
    tr_bytes = 2 * N_IMAGES * px + 2 * px * 4 * K  # T_B = 2 n P b + 2 P D
    re_bytes = 2 * N_IMAGES * px + px * (2 + 4 + 4)  # R_B = 2 n P b + P (2 + 4 + c)
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f)
    except OSError:
        pass
    # the same frames one match after the other on one stream: every kernel alone on the GPU
    h.set_overlap(False)
    for _ in range(2):
        step_serial()
    torch.cuda.synchronize()
    h.set_profiling(True)
    ev0.record()
    for _ in range(5):
        step_serial()
    ev1.record()
    alone_ms, alone_n = h.stage_times()
    h.set_profiling(False)
    serial_ms_per_match = ev0.elapsed_time(ev1) / (5 * FRAMES)
    a_tr, a_se, a_re = (1e-3 * v / max(alone_n, 1) for v in alone_ms)

    # the other engine on the same frames, for the record (stage timer of the handle)
    engine = lb.search_engine()
    tensor = engine != "popc"  # K = 4, 2048 columns: inside the tensor-core engine's range
    lb.set_search_engine("popc" if tensor else "tensor")
    for _ in range(2):
        step_serial()
    torch.cuda.synchronize()
    h.set_profiling(True)
    for _ in range(3):
        step_serial()
    other_ms, other_n = h.stage_times()
    h.set_profiling(False)
    lb.set_search_engine(engine)
    h.set_overlap(True)
    t_other = 1e-3 * other_ms[1] / max(other_n, 1)
    t_popc, t_mma = (t_other, t_se) if tensor else (t_se, t_other)
    t_mma_alone = a_se if tensor else t_other

    popc_issued = COLS * px * 3  # the popc kernel's carry-save form: 3 POPC per 128-bit pair
    popc_line = {
        "kernel": "search_kernel<K=4, CONSISTENCY> (popc engine)", "bound": "popc", "achieved": popc_alg / t_popc / 1e12,
        "peak": popc_peak / 1e12, "unit": "Tpopc32/s", "frac": popc_alg / t_popc / popc_peak,
        "pipe_frac": popc_issued / t_popc / popc_peak, "traffic": traffic.get("search"),
        "peak_source": popc_src, "ms_per_launch": t_popc * 1e3,
        "note": "the integer-pipe engine (BICOS_B200_SEARCH_ENGINE=popc): frac = algorithmic popc32 (SURVEY 8d) over the "
                "measured POPC issue rate; 3 POPC are issued per 128-bit pair, pipe_frac is the share of the POPC pipe in use",
    }
    int8_peak, int8_src = measure_int8_peak()
    # Consistency: the two-pass kernels (mma1 / mma2) compute a full W x W x 128 product per row and direction; the
    # one-pass kernel (mma3, the default for this workload) takes both directions from ONE product
    onepass = search_kernel.startswith("mma3")
    dirs = 1 if onepass else 2
    # SURVEY 8d scores every left/right descriptor pair of a row ONCE, however often an implementation visits it:
    # `frac` is that algorithmic figure, `frac_executed` counts what the kernel issues (both directions)
    mma_ops_once = 2.0 * COLS * px * 32 * K
    mma_ops = mma_ops_once * dirs
    # shared-memory bytes per 128x128 tile. mma2: 16 KB operand reads, 8 KB expansion, 2 KB packed ring; mma3: 16 KB block
    # reads (the streamed operand goes to tensor memory), 1 KB packed ring, 2 KB block expansion + reduction per item / 16 tiles
    smem_bytes = (COLS / 128) * (px / 128) * dirs * (19 if onepass else 26) * 1024
    mma_line = {
        "kernel": search_kernel, "bound": "tensor", "achieved": mma_ops_once / t_mma / 1e12,
        "peak": int8_peak, "unit": "TOP/s", "frac": mma_ops_once / t_mma / 1e12 / int8_peak, "traffic": traffic.get("search_mma3" if onepass else "search_mma2"),
        "peak_kind": "dense int8 tensor rate (tcgen05 kind::i8)", "peak_source": int8_src, "ms_per_launch": t_mma * 1e3,
        "achieved_executed": mma_ops / t_mma / 1e12, "frac_executed": mma_ops / t_mma / 1e12 / int8_peak,
        "executed_over_algorithmic": dirs,
        # ms_per_launch / achieved / frac are the timed region's: there the kernel shares its SMs with the previous frame's
        # refine CTAs (match_batch). The same kernel with the GPU to itself (one match after the other, same run):
        "alone": {"ms_per_launch": t_mma_alone * 1e3, "achieved": mma_ops_once / t_mma_alone / 1e12,
                  "frac": mma_ops_once / t_mma_alone / 1e12 / int8_peak,
                  "achieved_executed": mma_ops / t_mma_alone / 1e12, "frac_executed": mma_ops / t_mma_alone / 1e12 / int8_peak},
        "smem_frac": smem_bytes / t_mma / (128.0 * 148 * sm_max * 1e6),
        # SURVEY 8d scores the search in popc32 (S = W * P * K) against the POPC pipe, the bound of a popcount kernel:
        # the same algorithmic work over this engine's time, for comparison with that table
        "algorithmic_popc32": {"achieved": popc_alg / t_mma / 1e12, "peak": popc_peak / 1e12, "unit": "Tpopc32/s",
                               "frac": popc_alg / t_mma / popc_peak, "peak_source": popc_src},
        "note": "the tensor-core engine (default): W x W x 128-bit Hamming matrix per row as int8 tcgen05.mma (kind::i8, TMEM "
                "accumulators), argmin in the epilogue. frac = 2*W*P*bits int8 ops (every descriptor pair once, SURVEY 8d) over "
                "the stage time and the dense int8 rate; frac_executed counts what the kernel issues: the same for the one-pass "
                "kernel (mma3: forward minima in-thread, reverse minima elementwise across the row's tiles, both from one "
                "product), twice that for the two-pass kernels (mma1 / mma2). The one-pass kernel is bound by the ALU pipe "
                "(the two folds), not by the tensor pipe: profiles/r02_ncu_search_mma_history.md. smem_frac: shared-memory "
                "bytes the kernel moves over 128 B/clk/SM",
    }
    roofline = mma_line if tensor else popc_line
    roofline["engine"] = "tensor" if tensor else "popc"
    roofline["other_engine"] = popc_line if tensor else mma_line
    roofline_other = [
        {"kernel": "transform_limited_kernel<u8,4> x2", "bound": "hbm", "achieved": tr_bytes / t_tr / 1e9,
         "peak": hbm_peak, "unit": "GB/s", "frac": tr_bytes / t_tr / 1e9 / hbm_peak, "traffic": traffic.get("transform"),
         "peak_source": hbm_src, "ms_per_launch": t_tr * 1e3 / 2},
        {"kernel": "refine_kernel<u8,float,subpixel,33>", "bound": "hbm", "achieved": re_bytes / t_re / 1e9,
         "peak": hbm_peak, "unit": "GB/s", "frac": re_bytes / t_re / 1e9 / hbm_peak, "traffic": traffic.get("refine"),
         "peak_source": hbm_src, "ms_per_launch": t_re * 1e3,
         "note": "subpixel mode is FP32-issue bound (20 x-steps x n x ~13 flops per pixel), not HBM bound"},
    ]

    cpu_baseline = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)  # the CPU reference gets every host core again
        t, kind, cores = cpu_reference_run(16)
        # the whole frame when that stays under a minute (16 host cores: about 6 s), else about 15 s of CPU work
        est = t / 16 * ROWS
        rows = ROWS if est <= 60.0 else int(min(ROWS, max(16, 16 * (15.0 / max(t, 1e-3)))))
        keep = {}
        t, kind, cores = cpu_reference_run(rows, keep=keep)
        cpu_baseline = {"value": rows * COLS / t / 1e6, "unit": "Mpx/s", "cores": cores, "kind": kind,
                        "sample": f"{rows} of {ROWS} rows of one stereo stack, {t:.1f} s wall, all host threads"}
        # the frame the timed region produced last (same kernels, same dispatch) against the reference's output
        parity = parity_against_reference(keep, timed_frame0[0], timed_frame0[1], kind)
        parity["search_kernel"] = search_kernel

    # the reference's own CUDA backend, unmodified, compiled for sm_100a (oracle/_ref/libbicos_refcuda.so):
    # a second baseline beside the CPU build (BASELINE.json north_star); device-resident inputs
    reference_cuda = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            import oracle

            if oracle.refcuda.available():
                l0, r0 = host[0]
                med, mn = oracle.refcuda.time(l0, r0, warmup=3, iters=9, **CFG)
                reference_cuda = {"value": px / med / 1e3, "unit": "Mpx/s", "ms_per_match": med, "ms_per_match_min": mn,
                                  "how": "unmodified reference src/impl/cuda.cu (BICOS_CUDA_HAS_UINT128) built for sm_100a "
                                         "against oracle/shim; median of 9 individually timed BICOS::match calls"}
        except Exception as e:  # a baseline must never take the product's numbers down with it
            reference_cuda = {"unavailable": str(e)}

    line = {
        "metric": "Mpx/s disparity", "value": value, "unit": "Mpx/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "ms_per_match": ms_per_step / FRAMES,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": CONFIG,
        "e2e": {"value": e2e_value, "unit": "Mpx/s", "h2d_bytes_per_step": FRAMES * 2 * N_IMAGES * px,
                "d2h_bytes_per_step": FRAMES * px * 8, "ms_per_step": e2e_ms, "matches_device_path": same, "host_affinity": affinity,
                "devices": devices, "device_policy": device_policy,
                "h2d_gbs": e2e_h2d_gbs, "link_gbs": link_gbs, "link_frac": e2e_h2d_gbs / link_gbs,
                "link_note": "link_gbs = plain 256 MB pinned host-to-device copies on the same GPUs, all ranks at once; the "
                             "device-to-host results (12 % of the bytes) travel the other direction of the link at the same time",
                "api": f"bicos_b200_match_host_begin/_end, {inflight} frames in flight (pinned host stacks -> host disparity + corrmap)"},
        "gpu_launches": launches,
        "stage_ms_per_match": {"transform_x2": t_tr * 1e3, "search": t_se * 1e3, "refine": t_re * 1e3,
                               "note": "CUDA events around each stage on its own stream inside the timed region; search and refine of "
                                       "consecutive frames overlap there, so the stages add up to more than ms_per_match"},
        "serial": {"ms_per_match": serial_ms_per_match, "mpx_per_s": px / serial_ms_per_match / 1e3,
                   "stage_ms_per_match": {"transform_x2": a_tr * 1e3, "search": a_se * 1e3, "refine": a_re * 1e3},
                   "note": "bicos_b200_match frame after frame on one stream (round 1's timed region): every kernel alone on the GPU"},
        "roofline": roofline, "roofline_other": roofline_other, "cpu_baseline": cpu_baseline, "parity": parity,
        "row_sharded": row_sharded, "reference_cuda": reference_cuda, "clocks": clocks,
    }
    print(json.dumps(line))
    if parity is not None and not parity["within_north_star"]:
        print(f"bench.py: PARITY FAILURE against the reference: {parity}", file=sys.stderr)
        sys.exit(3)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
