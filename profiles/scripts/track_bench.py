"""Pose tracking (ICP.track) on the cfg-2 room, 360 beams, course map.
   python profiles/scripts/track_bench.py [out.json]
Prints one JSON line (and writes it to out.json when given) with, from one process on one GPU:
- the card name and power limit (nvidia-smi);
- H = 1 from the true start over 300 scans taken one in six (room 9001): the call's time per scan by host clock
  (median of 3 after one untimed call) against the same loop run per scan from the host (process_scans for the
  odometry, then one map_observation per scan with the prior composed on the host), the error against the truth,
  and one stage's device work by CUDA events (median of 20 after 3 warm-up launches): the whole stage as the call
  enqueues it (virtual scan, replicate, ICP with score, track step) against its ICP alone; plus the B2S_TRACE
  timeline of an 8-scan call, from a child process;
- H = 27 324 (the whole 0.5 m / 10 deg grid of room 9001) at K = 1, 2, 4, 8: the time per call (host clock);
- over rooms 9002-9009, windows of 8 scans ending at every eighth scan (6 per room): how often the pose of the
  window's last scan lies within 0.10 m / 0.05 rad of the truth for the exhaustive relocalize of that scan alone,
  track over the last 4 and all 8 scans from the whole grid, and relocalize(first scan, keep=1024) followed by track
  over the 8 scans from the survivors, each with its time per window."""
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

N, EVERY, STREAM = 360, 6, 300
A0, A1 = -math.pi, math.pi
INC = (A1 - A0) / (N - 1)
QUALITY_SEEDS = range(9002, 9010)
WINDOWS = 6  # windows of 8 scans per quality room
TOL_XY, TOL_YAW = 0.10, 0.05


def events(fn, launches=20, warm=3):
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


def step(p, t):
    x, y, yaw = p
    c, s = math.cos(yaw), math.sin(yaw)
    return np.array([x + c * t[0, 2] - s * t[1, 2], y + s * t[0, 2] + c * t[1, 2], yaw + math.atan2(t[1, 0], t[0, 0])])


def errors(pose, truth):
    d_xy = np.hypot(pose[..., 0] - truth[..., 0], pose[..., 1] - truth[..., 1])
    d_yaw = np.abs((pose[..., 2] - truth[..., 2] + math.pi) % (2 * math.pi) - math.pi)
    return d_xy, d_yaw


def host_loop(icp, ranges, start):
    """The per-scan host loop the call replaces: odometry, then one map observation per scan at the composed prior."""
    odo, _ = icp.process_scans(ranges, A0, A1)
    pose = np.empty((len(ranges), 3))
    prior = np.asarray(start, dtype=np.float64)
    for k in range(len(ranges)):
        T, _ = icp.map_observation(ranges[k:k + 1], prior[None], A0, A1)
        pose[k] = step(prior, T[0])
        if k + 1 < len(ranges):
            prior = step(pose[k], odo[k])
    return pose


def stream_h1(icp, w):
    ranges, truth = w["ranges"][::EVERY], w["poses"][::EVERY]
    K = len(ranges)
    res = {"scans": K, "every": EVERY}
    res["track_per_scan_us"] = host(lambda: icp.track(ranges, truth[0], A0, A1)) * 1e3 / K
    res["host_loop_per_scan_us"] = host(lambda: host_loop(icp, ranges, truth[0])) * 1e3 / K
    best, pose, score, it, joint = icp.track(ranges, truth[0], A0, A1)
    loop = host_loop(icp, ranges, truth[0])
    res["host_loop_max_pose_diff"] = float(np.abs(loop - pose).max())
    d_xy, d_yaw = errors(pose, truth)
    res.update(err_xy_max=float(d_xy.max()), err_xy_mean=float(d_xy.mean()), err_yaw_max=float(d_yaw.max()),
               err_yaw_mean=float(d_yaw.mean()), iterations_mean=float(it.mean()))
    # one stage's device work, as the call enqueues it
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    obs = w["obstacles_course"]
    ox, oy, cs = cuda(obs[0]), cuda(obs[1]), cuda(scan.beam_table(A0, A1, N))
    prior, nxt, pose_d = cuda(truth[:1]), torch.empty((1, 3), dtype=torch.float64, device="cuda"), torch.empty(
        (1, 3), dtype=torch.float64, device="cuda")
    joint_d = torch.zeros(1, dtype=torch.float64, device="cuda")
    fin = torch.ones(1, dtype=torch.int32, device="cuda")
    odo = cuda(icp.process_scans(ranges[:2], A0, A1)[0][0])
    tar = torch.empty((1, 2, N), dtype=torch.float64, device="cuda")
    one = cuda(scan.laser_to_points(ranges[0], A0, A1)[:2][None])
    src = torch.empty_like(one)

    def stage():
        devapi.virtual_scan_batch(ox, oy, prior, A0, INC, N, beam_cs=cs, tar_xy=tar)
        src.copy_(one)
        T, _, err = devapi.icp_batch_err(tar, src)
        devapi.track_step(T, err, prior, pose_d, joint_d, fin, 1, odometry=odo, next_prior=nxt)
    res["stage_device_us"] = events(stage) * 1e3
    res["stage_icp_device_us"] = events(lambda: devapi.icp_batch_err(tar, src)) * 1e3
    # the B2S_TRACE timeline of an 8-scan call, in a child process (the variable is read per call)
    child = ("import sys, math, numpy as np; sys.path.insert(0, %r); import b2slam; from b2slam import synth;"
             "w = synth.room_relocalization(9001, 8 * %d, %d); icp = b2slam.ICP(); icp.set_static_map(w['obstacles_course']);"
             "r = w['ranges'][::%d]; icp.track(r, w['poses'][0], -math.pi, math.pi);"
             "icp.track(r, w['poses'][0], -math.pi, math.pi)") % (ROOT, EVERY, N, EVERY)
    env = dict(os.environ, B2S_TRACE="1")
    out = subprocess.run([sys.executable, "-c", child], env=env, capture_output=True, text=True, timeout=600)
    lines = [l for l in out.stderr.splitlines() if l.startswith("[b2s trace]")]
    res["trace_8_scans_second_call"] = lines[len(lines) // 2:]
    return res


def grid_timing(icp, w):
    cand = w["candidates"]
    ranges = w["ranges"][::EVERY]
    res = {"candidates": len(cand)}
    for K in (1, 2, 4, 8):
        res["K%d_ms" % K] = host(lambda: icp.track(ranges[:K], cand, A0, A1))
    res["relocalize_1_scan_ms"] = host(lambda: icp.relocalize(ranges[0], cand, A0, A1))
    return res


def quality(icp):
    hits = {"relocalize_1": 0, "track_K4": 0, "track_K8": 0, "keep1024_then_track_K8": 0}
    ms = {k: [] for k in hits}
    total = 0
    for seed in QUALITY_SEEDS:
        w = synth.room_relocalization(seed, 8 * WINDOWS * EVERY, N)
        icp.set_static_map(w["obstacles_course"])
        ranges, truth, cand = w["ranges"][::EVERY], w["poses"][::EVERY], w["candidates"]
        for win in range(WINDOWS):
            r, last = ranges[8 * win:8 * win + 8], truth[8 * win + 7]
            total += 1

            def judge(name, pose, t0):
                ms[name].append((time.perf_counter() - t0) * 1e3)
                d_xy, d_yaw = errors(pose, last)
                hits[name] += int(bool(d_xy < TOL_XY and d_yaw < TOL_YAW))
            t0 = time.perf_counter()
            best, pose, _, _ = icp.relocalize(r[7], cand, A0, A1)
            judge("relocalize_1", pose, t0)
            for K in (4, 8):
                t0 = time.perf_counter()
                best, pose, _, _, _ = icp.track(r[8 - K:], cand, A0, A1)
                judge("track_K%d" % K, pose[best, -1] if best >= 0 else np.full(3, np.nan), t0)
            t0 = time.perf_counter()
            _, _, _, _, kept = icp.relocalize(r[0], cand, A0, A1, keep=1024)
            best, pose, _, _, _ = icp.track(r, cand[kept], A0, A1)
            judge("keep1024_then_track_K8", pose[best, -1] if best >= 0 else np.full(3, np.nan), t0)
    return {"windows": total, "within": hits, "median_ms_per_window": {k: float(np.median(v)) for k, v in ms.items()}}


def main():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    out = {"card": card[0] if card else "unknown", "torch": torch.__version__}
    icp = b2slam.ICP()
    w = synth.room_relocalization(9001, STREAM * EVERY, N)
    icp.set_static_map(w["obstacles_course"])
    # (the quality rooms first: the whole call at the grid's size is warmed up there)
    out["quality"] = quality(icp)
    print("quality", json.dumps(out["quality"]), file=sys.stderr, flush=True)
    icp.set_static_map(w["obstacles_course"])
    out["stream_h1"] = stream_h1(icp, w)
    print("stream_h1", json.dumps(out["stream_h1"]), file=sys.stderr, flush=True)
    out["grid"] = grid_timing(icp, w)
    line = json.dumps(out)
    print(line)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
