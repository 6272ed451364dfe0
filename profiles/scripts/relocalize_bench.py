"""Relocalization (ICP.relocalize) on the cfg-2 room, seed 9001, 360 beams, course map.
   python profiles/scripts/relocalize_bench.py [out.json]
Prints one JSON line (and writes it to out.json when given) with, from one process on one GPU:
- the card name and power limit (nvidia-smi);
- for H = 1 000, 10 000 and 57 600 candidates (a seeded sample of synth.room_relocalization's grid at 0.25 m / 10 deg):
  the device work of one call split by CUDA events (median of 10 after 2 warm-up launches) into the H virtual scans
  (b2s_virtual_scan_batch), the H-pair ICP of one scan with its score (b2s_icp_batch_f64_err) and the selection
  (b2s_relocalize_select); the whole ICP.relocalize call on 8 scans by host clock (median of 5 after one untimed call),
  per scan; and the B2S_TRACE timeline of one 2-scan call, from which the per-scan segment (source cloud, its
  replication into the H rows and the ICP) is read against the ICP alone;
- the iteration histograms of right hypotheses (composed pose within 0.10 m and 0.05 rad of the truth) and wrong ones;
- on the full 0.5 m / 10 deg grid of room_relocalization(9001, 8, 360): each scan's chosen pose against the truth;
- the per-hypothesis host path (scan.virtual_scan + laser_to_points + ICP.process) on 200 hypotheses, host clock, and
  whether it gives relocalize's transforms."""
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import b2slam  # noqa: E402
from b2slam import _lib, devapi, scan, synth  # noqa: E402

N, SCANS = 360, 8
A0, A1 = -math.pi, math.pi
INC = (A1 - A0) / (N - 1)
SIZES = (1000, 10000, 57600)


def events(fn, launches=10, warm=2):
    ms = []
    for i in range(warm + launches):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        if i >= warm:
            ms.append(a.elapsed_time(b))
    return ms


def stat(ms):
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "n": len(ms)}


def candidates(count):
    grid = synth.room_relocalization(9001, 1, N, xy_step=0.25)["candidates"]
    rng = np.random.Generator(np.random.PCG64(count))
    return np.ascontiguousarray(grid[np.sort(rng.choice(grid.shape[0], count, replace=False))])


TRACE_CHILD = """
import math, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import b2slam
from b2slam import synth
w = synth.room_relocalization(9001, 2, 360)
cand = np.load(sys.argv[2])
icp = b2slam.ICP()
icp.set_static_map(w["obstacles_course"])
icp.relocalize(w["ranges"], cand, -math.pi, math.pi)
icp.relocalize(w["ranges"], cand, -math.pi, math.pi)
"""


def trace(cand, tmp):
    path = os.path.join(tmp, "cand.npy")
    np.save(path, cand)
    env = dict(os.environ, B2S_TRACE="1")
    err = subprocess.run([sys.executable, "-c", TRACE_CHILD, ROOT, path], env=env, capture_output=True,
                         text=True, check=True).stderr
    lines = [l for l in err.splitlines() if l.startswith("[b2s trace]")]
    return lines[len(lines) // 2:]  # the second call's timeline


def main():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    w = synth.room_relocalization(9001, SCANS, N)
    obs = w["obstacles_course"]
    out = {"workload": "cfg-2 room seed 9001, %d scans x %d beams, course map %d cells" % (SCANS, N, obs.shape[1]),
           "device": card[0] if card else None, "sizes": {}}
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")
    ox, oy, cs = cuda(obs[0]), cuda(obs[1]), cuda(scan.beam_table(A0, A1, N))
    icp = b2slam.ICP()
    icp.set_static_map(obs)
    tmp = tempfile.mkdtemp()
    for H in SIZES:
        cand = candidates(H)
        res = {}
        cd = cuda(cand)
        tar = torch.empty((H, 2, N), dtype=torch.float64, device="cuda")
        res["virtual_scans"] = stat(events(lambda: devapi.virtual_scan_batch(ox, oy, cd, A0, INC, N, beam_cs=cs,
                                                                             tar_xy=tar)))
        src1 = cuda(scan.laser_to_points(w["ranges"][0], A0, A1)[:2])
        src = src1[None].expand(H, 2, N).contiguous()
        T = torch.empty((H, 3, 3), dtype=torch.float64, device="cuda")
        it = torch.empty(H, dtype=torch.int32, device="cuda")
        err = torch.empty(H, dtype=torch.float64, device="cuda")
        res["icp_one_scan"] = stat(events(lambda: devapi.icp_batch_err(tar, src, 30, 1e-3, T, it, err)))
        res["icp_one_scan_without_score"] = stat(events(lambda: devapi.icp_batch(tar, src, 30, 1e-3, T, it)))
        sc = err[None].expand(SCANS, H).contiguous()
        Tk = T[None].expand(SCANS, H, 3, 3).contiguous()
        res["select_%d_scans" % SCANS] = stat(events(lambda: devapi.relocalize_select(sc, Tk, cd)))
        icp.relocalize(w["ranges"], cand, A0, A1)
        ms = []
        for _ in range(5):
            t = time.perf_counter()
            best, pose, score, iters, Th = icp.relocalize(w["ranges"], cand, A0, A1, return_T=True)
            ms.append((time.perf_counter() - t) * 1e3)
        res["call_%d_scans_host_clock" % SCANS] = dict(stat(ms), per_scan_ms=float(np.median(ms)) / SCANS)
        res["trace_2_scans"] = trace(cand, tmp)
        # right and wrong hypotheses: the composed pose of every hypothesis against the truth
        c, s = np.cos(cand[:, 2]), np.sin(cand[:, 2])
        px = cand[None, :, 0] + c * Th[..., 0, 2] - s * Th[..., 1, 2]
        py = cand[None, :, 1] + s * Th[..., 0, 2] + c * Th[..., 1, 2]
        pyaw = cand[None, :, 2] + np.arctan2(Th[..., 1, 0], Th[..., 0, 0])
        truth = w["poses"][:, None, :]
        right = (np.hypot(px - truth[..., 0], py - truth[..., 1]) < 0.10) & \
                (np.abs((pyaw - truth[..., 2] + math.pi) % (2 * math.pi) - math.pi) < 0.05)
        res["hypotheses_right"] = int(right.sum())
        res["iterations_histogram_right"] = np.bincount(iters[right], minlength=31).tolist()
        res["iterations_histogram_wrong"] = np.bincount(iters[~right], minlength=31).tolist()
        res["mean_iterations_right"] = float(iters[right].mean()) if right.any() else None
        res["mean_iterations_wrong"] = float(iters[~right].mean())
        d_xy = np.hypot(pose[:, 0] - w["poses"][:, 0], pose[:, 1] - w["poses"][:, 1])
        d_yaw = np.abs((pose[:, 2] - w["poses"][:, 2] + math.pi) % (2 * math.pi) - math.pi)
        res["best_pose_error_max_m"], res["best_pose_error_max_rad"] = float(d_xy.max()), float(d_yaw.max())
        out["sizes"][str(H)] = res
        del tar, src, T, it, err, sc, Tk
        torch.cuda.empty_cache()

    # the full 0.5 m / 10 deg grid of room_relocalization on its 8 scans: how far each chosen pose is from the truth
    best, pose, score, iters = icp.relocalize(w["ranges"], w["candidates"], A0, A1)
    out["full_grid"] = {"candidates": int(len(w["candidates"])),
                        "pose_error_m": np.hypot(pose[:, 0] - w["poses"][:, 0], pose[:, 1] - w["poses"][:, 1]).tolist(),
                        "pose_error_rad": np.abs((pose[:, 2] - w["poses"][:, 2] + math.pi) % (2 * math.pi)
                                                 - math.pi).tolist(),
                        "best_score": [float(score[k, b]) for k, b in enumerate(best)]}

    # the per-hypothesis host path on 200 hypotheses of scan 0
    cand = candidates(1000)[:200]
    _, _, _, _, Tb = icp.relocalize(w["ranges"][0], cand, A0, A1, return_T=True)

    def one(h):
        v = scan.virtual_scan(obs, cand[h], A0, INC, N)
        return icp.process(scan.laser_to_points(v, A0, A1), scan.laser_to_points(w["ranges"][0], A0, A1))
    for h in range(20):
        one(h)
    t = time.perf_counter()
    Ts = np.stack([one(h) for h in range(200)])
    per_us = (time.perf_counter() - t) * 1e6 / 200
    out["per_hypothesis_host_path"] = {"hypotheses": 200, "per_hypothesis_us": per_us,
                                       "transforms_byte_identical": bool(Ts.tobytes() == Tb.tobytes())}
    line = json.dumps(out)
    print(line)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
