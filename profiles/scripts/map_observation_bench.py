"""Map observation of W9 localization (calc_map_observation, [LOC9]:152-157) on the cfg-2 room, seed 9001.
   python profiles/scripts/map_observation_bench.py [out.json]
Prints one JSON line (and writes it to out.json when given) with, from one process on one GPU:
- the card name and power limit (nvidia-smi) and b2s_measure_fp64_peak;
- the batched virtual-scan kernel alone (b2s_virtual_scan_batch writing the ICP target, as the map observation runs
  it): CUDA events around each launch, median of 30 after 3 warm-up launches, for 9 999 poses x 360 beams on the
  course map (129^2 cells at 0.155 m) and on the fine map (2600^2 at 0.01 m, > 2e5 cells); obstacle evaluations/s and
  the FP64-pipe share they imply at the instructions per evaluation counted in the SASS
  (profiles/r6/sass/virtual_scan_batch_obstacle_loop.sass);
- the ICP solve alone on the same 9 999 target / source pairs (b2s_icp_batch_f64, CUDA events, median of 30);
- the whole ICP.map_observation call: host clock around the synchronised call with page-locked inputs, median of 30
  after >= 50 ms of untimed calls (first calls pay allocation and module loading), at the automatic pipeline depth
  and at forced depths (b2s_tune h2d_chunks), on 9 999 and on 3 000 scans;
- the per-scan path of today on the first 200 scans: scan.virtual_scan + laser_to_points + ICP.process per scan, host
  clock over the 200 after 20 untimed scans, reported per scan; and whether it gives the batched call's bytes."""
import ctypes
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
from b2slam import _lib, devapi, scan, synth  # noqa: E402

# FP64-pipe instructions per obstacle evaluation in the obstacle loop of virtual_scan_batch_kernel (the SASS above):
# 59 DFMA / DMUL / DADD, 12 DSETP, 3 MUFU.*64H.  Of the 59: hypot 17 (with the four differences), atan2 32, the
# bin expression 10.
FP64_PER_EVAL, DFMA_CLASS_PER_EVAL = 74, 59
K, N = 9999, 360
A0, A1 = -math.pi, math.pi
INC = (A1 - A0) / (N - 1)


def events(fn, launches=30, warm=3):
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


def host_clock(fn, calls=30, warm_s=0.05):
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < warm_s:
        fn()
    ms = []
    for _ in range(calls):
        t = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t) * 1e3)
    return ms


def main():
    L = _lib.lib()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    peak = ctypes.c_double(0.0)
    _lib.check(L.b2s_measure_fp64_peak(ctypes.byref(peak)))
    peak_tflops = peak.value
    room = synth.room_map_observation(9001, K, N)
    maps = {"course": room["obstacles_course"], "fine": room["obstacles_fine"]}
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")
    poses = cuda(room["prior"])
    cs = cuda(scan.beam_table(A0, A1, N))
    tar = torch.empty((K, 2, N), dtype=torch.float64, device="cuda")
    out = {"workload": "cfg-2 room seed 9001, %d scans x %d beams, prior poses; course map %d cells, fine map %d cells"
           % (K, N, maps["course"].shape[1], maps["fine"].shape[1]),
           "device": card[0] if card else None, "fp64_peak_tflops_same_run": peak_tflops,
           "fp64_pipe_instructions_per_evaluation": FP64_PER_EVAL,
           "dfma_class_instructions_per_evaluation": DFMA_CLASS_PER_EVAL}

    # --- the virtual-scan kernel alone
    for name, obs in maps.items():
        ox, oy = cuda(obs[0]), cuda(obs[1])
        ms = events(lambda: devapi.virtual_scan_batch(ox, oy, poses, A0, INC, N, beam_cs=cs, tar_xy=tar))
        evals = K * obs.shape[1]
        rate = evals / (np.median(ms) * 1e-3)
        out["vscan_kernel_" + name] = dict(stat(ms), obstacles=int(obs.shape[1]), evaluations=evals,
                                           evaluations_per_s=rate,
                                           # DFMA-class instructions against the DFMA issue rate (peak / 2 flop)
                                           dfma_pipe_share=rate * DFMA_CLASS_PER_EVAL / (peak_tflops * 1e12 / 2))

    # --- the ICP solve alone on the course map's targets
    ox, oy = cuda(maps["course"][0]), cuda(maps["course"][1])
    devapi.virtual_scan_batch(ox, oy, poses, A0, INC, N, beam_cs=cs, tar_xy=tar)
    src = cuda(np.stack([scan.laser_to_points(r, A0, A1)[:2] for r in room["ranges"]]))
    T_d = torch.empty((K, 3, 3), dtype=torch.float64, device="cuda")
    it_d = torch.empty(K, dtype=torch.int32, device="cuda")
    out["icp_solve_course"] = stat(events(lambda: devapi.icp_batch(tar, src, 30, 1e-3, T_d, it_d)))

    # --- the whole host call
    icp = b2slam.ICP()
    ranges_p = _lib.pinned_empty((K, N), np.float32)
    ranges_p[:] = room["ranges"]
    prior_p = _lib.pinned_empty((K, 3), np.float64)
    prior_p[:] = room["prior"]
    for name, obs in maps.items():
        icp.set_static_map(obs)
        res = {}
        for chunks in (0, 1, 2, 4, 8):
            _lib.check(L.b2s_tune(b"h2d_chunks", chunks))
            for k in (K, 3000):
                ms = host_clock(lambda: icp.map_observation(ranges_p[:k], prior_p[:k], A0, A1))
                res["scans%d_chunks%s" % (k, chunks or "auto")] = dict(stat(ms), per_scan_us=float(np.median(ms)) * 1e3 / k)
        _lib.check(L.b2s_tune(b"h2d_chunks", 0))
        out["map_observation_call_" + name] = res

    # --- today's per-scan path, 200 scans of the course map
    icp.set_static_map(maps["course"])
    T_b, it_b = icp.map_observation(room["ranges"][:200], room["prior"][:200], A0, A1)

    def per_scan(k):
        v = scan.virtual_scan(maps["course"], room["prior"][k], A0, INC, N)
        return icp.process(scan.laser_to_points(v, A0, A1), scan.laser_to_points(room["ranges"][k], A0, A1))
    for k in range(20):
        per_scan(k)
    t = time.perf_counter()
    T_s = np.stack([per_scan(k) for k in range(200)])
    per_ms = (time.perf_counter() - t) * 1e3 / 200
    batched = out["map_observation_call_course"]["scans%d_chunksauto" % K]["per_scan_us"]
    out["per_scan_path_course"] = {"scans": 200, "per_scan_us": per_ms * 1e3,
                                   "batched_per_scan_us": batched, "speedup_per_scan": per_ms * 1e3 / batched,
                                   "transforms_byte_identical": bool(T_s.tobytes() == T_b.tobytes())}
    line = json.dumps(out)
    print(line)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
