"""world_size-2 gloo run of the multi-GPU host logic on CPU tensors (SURVEY.md section 8e).

The per-rank ray-casts are done by the CPU oracle here (this is a test of the sharding and
merge plumbing, not of the kernels): rank-sharded count deltas summed by all_reduce must be
bit-identical to one pass over all streams, and gathered transforms must keep pair order."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    # CPU tensors only: with GPUs visible, init() would bind rank r to GPU r, which a one-GPU machine lacks for rank 1
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="")
    import b2slam.dist as bdist
    import b2slam.synth as synth
    from oracle import corc
    r, _, w = bdist.init(backend="gloo")
    assert (r, w) == (rank, world)
    G, S, H = 256, 10.0, 12.8
    streams = 4
    lo, hi = bdist.shard_bounds(streams, rank, world)
    hit = np.zeros((G, G), dtype=np.int32)
    miss = np.zeros((G, G), dtype=np.int32)
    for s in range(lo, hi):
        ox, oy, cx, cy = synth.grid_scans(5001 + s, 6, 120, half_extent_m=6.0)
        corc.grid_raycast(hit, miss, S, H, H, ox, oy, cx, cy)
    th, tm = torch.from_numpy(hit), torch.from_numpy(miss)
    bdist.allreduce_counts(th, tm)
    # transforms: each rank owns a block of 5 "pairs" tagged with their global index
    plo, phi = bdist.shard_bounds(5, rank, world)
    T = torch.zeros((phi - plo, 3, 3), dtype=torch.float64)
    for i in range(plo, phi):
        T[i - plo] = float(i)
    counts = [b - a for a, b in (bdist.shard_bounds(5, q, world) for q in range(world))]
    allT = bdist.gather_transforms(T, counts)
    slow = bdist.max_over_ranks(float(rank + 1), device="cpu")
    bdist.barrier()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), hit=th.numpy(), miss=tm.numpy(),
             T=allT.numpy(), slow=slow)
    dist.destroy_process_group()


def test_two_rank_grid_merge_and_gather(tmp_path):
    world = 2
    port = 29640 + (os.getpid() % 200)
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    import b2slam.synth as synth
    from oracle import corc
    G, S, H = 256, 10.0, 12.8
    hit = np.zeros((G, G), dtype=np.int32)
    miss = np.zeros((G, G), dtype=np.int32)
    for s in range(4):
        ox, oy, cx, cy = synth.grid_scans(5001 + s, 6, 120, half_extent_m=6.0)
        corc.grid_raycast(hit, miss, S, H, H, ox, oy, cx, cy)
    assert hit.sum() > 0
    for r in range(world):
        z = np.load(os.path.join(str(tmp_path), "rank%d.npz" % r))
        assert np.array_equal(z["hit"], hit) and np.array_equal(z["miss"], miss)
        assert [int(t[0, 0]) for t in z["T"]] == [0, 1, 2, 3, 4]
        assert float(z["slow"]) == 2.0
