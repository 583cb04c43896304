"""Host-side multi-GPU logic on CPU: world_size-2 gloo processes, the oracle standing in for the
CUDA matcher (the oracle is allowed here: this is a test)."""

import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from libbicos_b200 import sharding, synth  # noqa: E402

KW = dict(nxcorr_threshold=0.9, subpixel_step=0.25, min_variance=1.0, consistency=True, max_lr_diff=1)
N, ROWS, COLS = 9, 37, 96  # odd row count: uneven blocks


def test_row_ranges_cover_exactly():
    for rows in (1, 7, 37, 1536):
        for world in (1, 2, 3, 8):
            blocks = [sharding.row_range(r, world, rows) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == rows
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1
    assert sum(len(sharding.frame_indices(r, 8, 256)) for r in range(8)) == 256


def _worker(rank, world, port, tmp):
    sys.path.insert(0, ROOT)
    import oracle

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        def match_fn(s0, s1):
            d, c = oracle.port.match(s0.numpy(), s1.numpy(), **KW)
            return torch.from_numpy(d), torch.from_numpy(c)

        # row-sharded single match: every rank generates only its own rows
        lo, hi = sharding.row_range(rank, world, ROWS)
        l, r, _ = synth.make_stacks(N, ROWS, COLS, np.uint8, seed=21, row0=lo, rows=hi - lo)
        disp, corr = sharding.match_row_sharded(match_fn, torch.from_numpy(l), torch.from_numpy(r), ROWS)
        if rank == 0:
            np.save(os.path.join(tmp, "disp.npy"), disp.numpy())
            np.save(os.path.join(tmp, "corr.npy"), corr.numpy())
        else:
            assert disp is None and corr is None

        # frame-sharded batch: no communication, every frame done exactly once
        def load(f):
            a, b, _ = synth.make_stacks(N, 12, COLS, np.uint8, seed=21, frame=f)
            return torch.from_numpy(a), torch.from_numpy(b)

        done = sharding.match_frames_sharded(match_fn, load, 5)
        np.save(os.path.join(tmp, f"frames_{rank}.npy"), np.array([f for f, _, _ in done]))
        for f, d, _ in done:
            np.save(os.path.join(tmp, f"frame_{f}.npy"), d.numpy())
    finally:
        dist.destroy_process_group()


def test_row_and_frame_sharding_world2(tmp_path, oracles):
    world = 2
    port = 29500 + os.getpid() % 2000
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    l, r, _ = synth.make_stacks(N, ROWS, COLS, np.uint8, seed=21)
    want_d, want_c = oracles.port.match(l, r, **KW)
    assert np.array_equal(np.load(tmp_path / "disp.npy"), want_d, equal_nan=True)
    assert np.array_equal(np.load(tmp_path / "corr.npy"), want_c, equal_nan=True)
    frames = sorted(int(f) for k in range(world) for f in np.load(tmp_path / f"frames_{k}.npy"))
    assert frames == [0, 1, 2, 3, 4]
    for f in frames:
        a, b, _ = synth.make_stacks(N, 12, COLS, np.uint8, seed=21, frame=f)
        assert np.array_equal(np.load(tmp_path / f"frame_{f}.npy"), oracles.port.match(a, b, **KW)[0], equal_nan=True)


# ------------------------------------------------------------------ GPUs: NCCL + peer memory --
def _gpu_worker(rank, world, port, tmp):
    sys.path.insert(0, ROOT)
    import libbicos_b200 as lb

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        cfg = lb.Config(**KW)
        h = lb.Handle(rank)
        rows, cols, n = 203, 320, 33  # uneven blocks
        lo, hi = sharding.row_range(rank, world, rows)
        l, r, _ = synth.make_stacks(n, rows, cols, np.uint8, seed=33, row0=lo, rows=hi - lo, xp=torch, device="cuda")
        # (1) kernels store their rows into rank 0's images over NVLink peer memory
        pa = sharding.PeerAssembly(h, rows, cols, cfg, rank)
        for _ in range(2):  # reuse of the mapping
            pa.match(l, r)
            pd, pc = pa.finish()
        # (2) the same through a NCCL gather
        gd, gc = sharding.match_row_sharded(lambda a, b: h.match(a, b, cfg), l, r, rows)
        if rank == 0:
            np.save(os.path.join(tmp, "peer_disp.npy"), pd.cpu().numpy())
            np.save(os.path.join(tmp, "peer_corr.npy"), pc.cpu().numpy())
            np.save(os.path.join(tmp, "gather_disp.npy"), gd.cpu().numpy())
            np.save(os.path.join(tmp, "gather_corr.npy"), gc.cpu().numpy())
        else:
            assert pd is None and gd is None
        pa.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_row_sharded_match_on_two_gpus(tmp_path, oracles):
    """World size 2 over NCCL on real GPUs: peer-memory assembly and gather both equal the oracle."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = 2
    port = 29600 + os.getpid() % 2000
    mp.spawn(_gpu_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    l, r, _ = synth.make_stacks(33, 203, 320, np.uint8, seed=33)
    want_d, want_c = oracles.port.match(l, r, **KW)
    for kind in ("peer", "gather"):
        assert np.array_equal(np.load(tmp_path / f"{kind}_disp.npy"), want_d, equal_nan=True), kind
        assert np.array_equal(np.load(tmp_path / f"{kind}_corr.npy"), want_c, equal_nan=True), kind


def test_topology_pick_is_a_pure_function_of_the_matrix():
    """libbicos_b200.topology.choose: ranks spread over the PCIe tree NVML reports; every rank computes the same list."""
    from libbicos_b200 import topology

    def level(i, j):  # an HGX-like tree: GPU pairs on a switch, two switches per host bridge, two bridges
        return 0 if i == j else 10 if i // 2 == j // 2 else 30 if i // 4 == j // 4 else 50

    tree = [[level(i, j) for j in range(8)] for i in range(8)]
    assert topology.choose(2, tree)[0] == [0, 4]
    assert topology.choose(4, tree)[0] == [0, 2, 4, 6]
    flat = [[0 if i == j else 50 for j in range(8)] for i in range(8)]
    assert topology.choose(4, flat)[0] == [0, 2, 4, 6] and "flat" in topology.choose(4, flat)[1]
    assert topology.spread(2, 8) == [0, 4] and topology.spread(8, 8) == list(range(8))
    assert isinstance(topology.describe(), dict)  # without NVML: {"unavailable": ...}
