"""Coarse-to-fine relocalization (ICP.relocalize(keep=...)) against the exhaustive call, cfg-2 room, 360 beams, course
map.
   python profiles/scripts/relocalize_keep_bench.py [out.json]
Prints one JSON line (and writes it to out.json when given) with, from one process on one GPU:
- the card name and power limit (nvidia-smi);
- for the round-8 samples of H = 10 000 and 57 600 candidates (seed 9001, 0.25 m / 10 deg grid) and the whole
  0.125 m / 10 deg grid of room_relocalization(9001, ...): the exhaustive call and the staged call at every
  coarse_iters in COARSE x keep in KEEP on 8 scans, by host clock (median of 3 after one untimed call), per scan; and
  the device work split by CUDA events (median of 5 after 2 warm-up launches): the coarse H-pair ICP of one scan with
  its score (b2s_icp_batch_f64_err at max_iter = coarse_iters), the keep step over 8 scans (b2s_relocalize_keep), the
  refinement of the 8 x keep survivors (b2s_icp_batch_f64_err at max_iter = 30, one launch) and the selection among
  them (b2s_relocalize_select_kept);
- quality on room seeds 9002-9009 (8 scans each, each room's full 0.5 m / 10 deg grid) for every configuration: pose
  error against the truth, pose difference from the exhaustive result, the score gap to the exhaustive winner, and
  whether the exhaustive winner survived the keep step."""
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import b2slam  # noqa: E402
from b2slam import devapi, scan, synth  # noqa: E402

N, SCANS = 360, 8
A0, A1 = -math.pi, math.pi
INC = (A1 - A0) / (N - 1)
COARSE = (2, 3, 4, 5, 6, 8)
KEEP = (64, 256, 1024)
QUALITY_SEEDS = range(9002, 9010)


def events(fn, launches=5, warm=2):
    ms = []
    for i in range(warm + launches):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        if i >= warm:
            ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def host(fn, runs=3):
    fn()
    ms = []
    for _ in range(runs):
        t = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t) * 1e3)
    return float(np.median(ms))


def sample(count):  # the round-8 sampler (relocalize_bench.py)
    grid = synth.room_relocalization(9001, 1, N, xy_step=0.25)["candidates"]
    rng = np.random.Generator(np.random.PCG64(count))
    return np.ascontiguousarray(grid[np.sort(rng.choice(grid.shape[0], count, replace=False))])


def wrap(a):
    return np.abs((a + math.pi) % (2 * math.pi) - math.pi)


def timing(icp, w, cand):
    H = len(cand)
    res = {"candidates": H}
    ex = host(lambda: icp.relocalize(w["ranges"], cand, A0, A1))
    res["exhaustive_per_scan_ms"] = ex / SCANS
    # device splits
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")
    obs = w["obstacles_course"]
    ox, oy, cs, cd = cuda(obs[0]), cuda(obs[1]), cuda(scan.beam_table(A0, A1, N)), cuda(cand)
    tar = torch.empty((H, 2, N), dtype=torch.float64, device="cuda")
    devapi.virtual_scan_batch(ox, oy, cd, A0, INC, N, beam_cs=cs, tar_xy=tar)
    srcs = [cuda(scan.laser_to_points(w["ranges"][k], A0, A1)[:2]) for k in range(SCANS)]
    src = srcs[0][None].expand(H, 2, N).contiguous()
    T1 = torch.empty((SCANS, H, 3, 3), dtype=torch.float64, device="cuda")
    it1 = torch.empty((SCANS, H), dtype=torch.int32, device="cuda")
    e1 = torch.empty((SCANS, H), dtype=torch.float64, device="cuda")
    keys = torch.empty(SCANS * H, dtype=torch.int64, device="cuda")
    res["configs"] = {}
    for coarse in COARSE:
        # the coarse ICP of every scan (the keep step needs all 8); scan 0 timed
        for k in range(SCANS):
            s = srcs[k][None].expand(H, 2, N).contiguous()
            devapi.icp_batch_err(tar, s, coarse, 1e-3, T1[k], it1[k], e1[k])
            del s
        coarse_ms = events(lambda: devapi.icp_batch_err(tar, src, coarse, 1e-3, T1[0], it1[0], e1[0]))
        for keep in KEEP:
            M = min(keep, H)
            cfg = {"coarse_icp_one_scan_ms": coarse_ms}
            kept = devapi.relocalize_keep(e1, T1, keep, keys=keys)
            cfg["keep_8_scans_ms"] = events(lambda: devapi.relocalize_keep(e1, T1, keep, kept_out=kept, keys=keys))
            tar2 = tar[kept.reshape(-1).long()].contiguous()
            src2 = torch.stack([srcs[k][None].expand(M, 2, N) for k in range(SCANS)]).reshape(SCANS * M, 2, N).contiguous()
            T2 = torch.empty((SCANS * M, 3, 3), dtype=torch.float64, device="cuda")
            it2 = torch.empty(SCANS * M, dtype=torch.int32, device="cuda")
            e2 = torch.empty(SCANS * M, dtype=torch.float64, device="cuda")
            cfg["refine_8_scans_ms"] = events(lambda: devapi.icp_batch_err(tar2, src2, 30, 1e-3, T2, it2, e2))
            cfg["select_8_scans_ms"] = events(lambda: devapi.relocalize_select(
                e2.reshape(SCANS, M), T2.reshape(SCANS, M, 3, 3), cd, kept=kept))
            staged = host(lambda: icp.relocalize(w["ranges"], cand, A0, A1, keep=keep, coarse_iters=coarse))
            cfg["staged_per_scan_ms"] = staged / SCANS
            cfg["speedup"] = ex / staged
            res["configs"]["c%d_k%d" % (coarse, keep)] = cfg
            del tar2, src2, T2, it2, e2
    del tar, src, T1, it1, e1, keys
    torch.cuda.empty_cache()
    return res


def quality():
    per = {"c%d_k%d" % (c, k): {"pose_error_m": [], "pose_error_rad": [], "diff_from_exhaustive_m": [],
                                "diff_from_exhaustive_rad": [], "score_gap": [], "winner_survived": []}
           for c in COARSE for k in KEEP}
    ex_err = {"pose_error_m": [], "pose_error_rad": []}
    for seed in QUALITY_SEEDS:
        w = synth.room_relocalization(seed, SCANS, N)
        icp = b2slam.ICP()
        icp.set_static_map(w["obstacles_course"])
        truth = w["poses"]
        xb, xp, xs, _ = icp.relocalize(w["ranges"], w["candidates"], A0, A1)
        ex_err["pose_error_m"] += np.hypot(*(xp[:, :2] - truth[:, :2]).T).tolist()
        ex_err["pose_error_rad"] += wrap(xp[:, 2] - truth[:, 2]).tolist()
        for c in COARSE:
            for k in KEEP:
                b, p, s, _, kept = icp.relocalize(w["ranges"], w["candidates"], A0, A1, keep=k, coarse_iters=c)
                q = per["c%d_k%d" % (c, k)]
                q["pose_error_m"] += np.hypot(*(p[:, :2] - truth[:, :2]).T).tolist()
                q["pose_error_rad"] += wrap(p[:, 2] - truth[:, 2]).tolist()
                q["diff_from_exhaustive_m"] += np.hypot(*(p[:, :2] - xp[:, :2]).T).tolist()
                q["diff_from_exhaustive_rad"] += wrap(p[:, 2] - xp[:, 2]).tolist()
                q["score_gap"] += [float(s[i, list(kept[i]).index(b[i])] - xs[i, xb[i]]) if b[i] >= 0 else math.inf
                                   for i in range(SCANS)]
                q["winner_survived"] += [bool(xb[i] in kept[i]) for i in range(SCANS)]
        del icp
    summary = {"exhaustive": {"max_pose_error_m": max(ex_err["pose_error_m"]),
                              "max_pose_error_rad": max(ex_err["pose_error_rad"]),
                              "scans_within_0.10m_0.05rad": int(sum(a < 0.10 and b < 0.05 for a, b in
                                                                    zip(ex_err["pose_error_m"], ex_err["pose_error_rad"])))}}
    for name, q in per.items():
        summary[name] = {"scans": len(q["winner_survived"]),
                         "winner_survived": int(sum(q["winner_survived"])),
                         "same_pose_as_exhaustive": int(sum(d == 0.0 for d in q["diff_from_exhaustive_m"])),
                         "scans_within_0.10m_0.05rad": int(sum(a < 0.10 and b < 0.05 for a, b in
                                                               zip(q["pose_error_m"], q["pose_error_rad"]))),
                         "max_pose_error_m": max(q["pose_error_m"]), "max_pose_error_rad": max(q["pose_error_rad"]),
                         "max_diff_from_exhaustive_m": max(q["diff_from_exhaustive_m"]),
                         "max_score_gap": max(q["score_gap"])}
    return summary


def main():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    w = synth.room_relocalization(9001, SCANS, N)
    out = {"workload": "cfg-2 room seed 9001, %d scans x %d beams, course map" % (SCANS, N),
           "device": card[0] if card else None, "timing": {}}
    icp = b2slam.ICP()
    icp.set_static_map(w["obstacles_course"])
    fine = np.ascontiguousarray(synth.room_relocalization(9001, 1, N, xy_step=0.125)["candidates"])
    for name, cand in (("10000", sample(10000)), ("57600", sample(57600)), ("grid_0.125m", fine)):
        out["timing"][name] = timing(icp, w, cand)
        print(name, json.dumps(out["timing"][name]), file=sys.stderr, flush=True)
    out["quality_seeds_9002_9009"] = quality()
    line = json.dumps(out)
    print(line)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
