#!/usr/bin/env python
"""bench.py -- headline measurement of the b2slam hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--workload grid|icp] [--impl reference]

One JSON line on stdout (rank 0).  The primary workload is cfg 3 of BASELINE.json, the W12
occupancy-grid update (4096x4096 cells at 5 cm, 1080-beam scans, known poses), because it is the
half of the metric the HBM roofline target applies to; the same line carries the cfg 2 ICP
measurement (9 999 consecutive 360-beam pairs) under "icp".  `--workload icp` swaps the roles.

A step is one pass of the hot path over one batch of synthetic scans resident in HBM:
  grid: zero the count planes, ray-cast SCANS x 1080 beams, (N>1: merge the int32 count deltas
        over NVLink peer memory, or all-reduce them over NCCL with --merge nccl), finalize to the
        int8 occupancy map
  icp : ICP.process over the whole batch of pairs (one CTA per pair)
`e2e` is the same step through the host-buffer API with pinned host arrays in and the int8 occupancy map out, every
copy inside the timed region, after untimed calls that bring the GPU back to full clocks.  For the grid the headline is
the streaming form of the raw-scan call (dist.ShardedMappingP2P.submit_scans + Ticket.wait, two steps in flight: the
upload of step k+1 overlaps the read-back of step k; ranges + poses, 4 B per beam); beside it `e2e_blocking_call`
(Mapping.update_batch on world-frame endpoints, one call at a time; N > 1: ShardedMappingP2P.update_batch) and
`e2e_fused_ingestion` (the blocking raw-scan call Mapping.update_scans / ShardedMappingP2P.update_scans).  For the ICP
`e2e` is the streaming raw-range call too (ICP.submit_scans + IcpTicket.wait: cfg 2 is a scan stream), with
`e2e_streaming_sequence` (the same on float32 points, twice the bytes: PCIe-bound), `e2e_blocking_call`
(ICP.process_sequence), `e2e_fused_ingestion` (ICP.process_scans, blocking) and `e2e_pair_form` (ICP.process_batch on
explicit pairs, four times the bytes).

With N > 1 ranks the line also carries `merge_bit_identical`: after the timed region a reduced batch per rank goes
through the same peer-memory merge, every rank ray-casts ALL ranks' scans in one pass by itself, and the merged map
and its shard of the merged counts are compared byte for byte (all ranks must agree).  `cfg4` / `cfg5` hold the two
sharded configurations of BASELINE.json (1 M independent 1080-beam ICP pairs; a 16384 x 16384 grid from 8 scan
streams), strong scaling over the N ranks, each with a parity sample.

`--impl reference` times the reference's own CPU algorithm (the literal Python/NumPy port in
oracle/pyref.py -- the reference is pure Python, so there is nothing faster to be fair to) on
all host cores, on a bounded sample of the same workload.

`--dump-outputs DIR` writes, as DIR/<name>.npy (float64), what the last timed step of each measured path left for
its caller (rank 0's share with N > 1): the grid's count planes and occupancy map (cfg 5: the map), each as one
fixed, seeded sample of cells plus the sum of every row, and the ICP transforms and iteration counts (cfg 4: a fixed,
seeded sample of the pairs).  The inputs are seeded, so two builds run with the same arguments can be compared file
for file.
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GRID_CELLS = 4096
GRID_RESO = 0.05
GRID_BEAMS = 1080
ICP_BEAMS = 360
ICP_SCANS = 10000
FP64_PEAK_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12  # nominal B200 vector FP64 (no measured figure)
DUMP_CELLS = 1 << 19          # cells sampled from each map plane by --dump-outputs
DUMP_PAIRS = 1 << 16          # cfg-4 pairs sampled by --dump-outputs
DUMP_MAX_BYTES = 64 << 20     # all files of --dump-outputs together


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_stamp(key):
    """Figures that only a profiler can give (DRAM bytes, executed-instruction counts), taken from the committed ncu
    capture of this workload and stamped with the SHA-1 of the kernel sources they were measured on
    (profiles/r2/ncu_stamps.json, written by profiles/scripts/stamp_ncu.py).  A kernel edited since then makes the
    stamp stale: the entry is returned as None instead of quoting a number that belongs to other code."""
    import hashlib
    try:
        with open(os.path.join(ROOT, "profiles", "r2", "ncu_stamps.json")) as fh:
            ent = json.load(fh)[key]
        h = hashlib.sha1()
        for rel in ent["sources"]:
            with open(os.path.join(ROOT, rel), "rb") as fh:
                h.update(fh.read())
        return ent if h.hexdigest() == ent["sha1"] else None
    except Exception:
        return None


# =============================================================================== --dump-outputs

def seeded_sample(n, k, seed):
    """Sorted indices of a fixed, seeded sample of k of n elements (all n when k >= n)."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def keep_output(args, name, arr):
    """Hold one output (a device tensor) of a timed step for --dump-outputs, as float64 on the host."""
    args.outputs[name] = arr.cpu().numpy().astype(np.float64)


def keep_grid_outputs(args, prefix, planes, seed):
    """Grid outputs (2-D device tensors of one shape): every plane at the same seeded sample of cells, and the sum of
    each of its rows, so that a change in any cell shows while the files stay small."""
    import torch
    first = next(iter(planes.values()))
    idx = seeded_sample(first.numel(), DUMP_CELLS, seed)
    args.outputs[prefix + "_cells"] = idx.astype(np.float64)
    idx = torch.from_numpy(idx).to(first.device)
    for name, plane in planes.items():
        keep_output(args, "%s_%s_sample" % (prefix, name), plane.reshape(-1)[idx])
        keep_output(args, "%s_%s_row_sums" % (prefix, name), plane.sum(dim=1, dtype=torch.int64))


def write_outputs(outputs, out_dir):
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs, more than the %d allowed" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


# =============================================================================== clocks

class ClockSampler(object):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None
            return
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _run(self):
        nv = self._nvml
        names = {}
        for attr in dir(nv):
            if attr.startswith("nvmlClocksEventReason") or attr.startswith("nvmlClocksThrottleReason"):
                val = getattr(nv, attr)
                if isinstance(val, int) and val and "All" not in attr:
                    names[val] = attr.replace("nvmlClocksEventReason", "").replace(
                        "nvmlClocksThrottleReason", "")
        getter = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
            nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                if getter:
                    bits = getter(self._h)
                    for b, nm in names.items():
                        if bits & b and nm not in ("GpuIdle", "None", "ApplicationsClocksSetting"):
                            self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.002)

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
               "samples": len(self.samples)}
        if self.samples:
            out["sm_mhz"] = float(statistics.median(self.samples))
        return out


# =============================================================================== CPU baseline

def _cpu_grid_worker(args):
    from oracle import pyref
    ox, oy, cx, cy = args
    S, Hx, Hy = pyref.grid_scale(GRID_CELLS, GRID_CELLS, GRID_RESO)
    hit = np.zeros((GRID_CELLS, GRID_CELLS), dtype=np.int32)
    miss = np.zeros((GRID_CELLS, GRID_CELLS), dtype=np.int32)
    visits = 0
    for k in range(ox.shape[0]):
        visits += pyref.grid_update_counts(hit, miss, ox[k].astype(np.float64), oy[k].astype(np.float64),
                                           float(cx[k]), float(cy[k]), S, Hx, Hy)
    return visits


def _cpu_icp_worker(args):
    from oracle import pyref
    tar, src = args
    iters = 0
    for p in range(tar.shape[0]):
        t = np.ones((3, tar.shape[2]))
        s = np.ones((3, src.shape[2]))
        t[:2] = tar[p]
        s[:2] = src[p]
        iters += pyref.icp_process(t, s, 30, 1e-3)[1]
    return iters


def _split(n, parts):
    parts = max(1, min(parts, n))
    edges = [n * i // parts for i in range(parts + 1)]
    return [(edges[i], edges[i + 1]) for i in range(parts) if edges[i + 1] > edges[i]]


def cpu_grid_rate(pool, cores, scans, data):
    """beams/s of the literal Python port on `scans` scans spread over `cores` processes."""
    ox, oy, cx, cy = data
    jobs = [(ox[a:b], oy[a:b], cx[a:b], cy[a:b]) for a, b in _split(scans, cores)]
    t0 = time.perf_counter()
    visits = sum(pool.map(_cpu_grid_worker, jobs))
    dt = time.perf_counter() - t0
    return scans * ox.shape[1] / dt, dt, visits


def cpu_icp_rate(pool, cores, pairs, tar, src):
    idx = np.linspace(0, tar.shape[0] - 1, pairs).astype(np.int64)
    jobs = [(tar[idx[a:b]], src[idx[a:b]]) for a, b in _split(pairs, cores)]
    t0 = time.perf_counter()
    iters = sum(pool.map(_cpu_icp_worker, jobs))
    dt = time.perf_counter() - t0
    return pairs / dt, dt, iters


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# =============================================================================== reference arm

def run_reference(args):
    """The reference's CPU algorithm on all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    from b2slam import synth
    cores = host_cores()
    steps, warmup = args.steps, args.warmup
    budget_s = 150.0 / max(1, steps + warmup)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        if args.workload == "grid":
            probe_scans = max(cores, 8)
            data = synth.grid_scans(12001, max(probe_scans, 4096), GRID_BEAMS)
            rate, _, _ = cpu_grid_rate(pool, cores, probe_scans, data)
            scans = int(min(4096, max(cores, rate * budget_s / GRID_BEAMS)))
            times = []
            for i in range(warmup + steps):
                r, dt, _ = cpu_grid_rate(pool, cores, scans, data)
                if i >= warmup:
                    times.append(dt)
            per_step = sum(times) / len(times)
            value = scans * GRID_BEAMS / per_step
            metric, unit = "grid_beam_updates_per_s", "beams/s"
            sample = "%d of the cfg-3 scans x %d beams per step, literal Python port over %d processes" % (
                scans, GRID_BEAMS, cores)
            config = {"workload": "cfg3 W12 occupancy grid 4096x4096 @ 0.05 m, 1080-beam scans, known poses",
                      "scans_per_step": scans, "beams": GRID_BEAMS}
        else:
            xy, _ = synth.room_sequence(9001, 513, ICP_BEAMS)
            tar, src = xy[:-1], xy[1:]
            rate, _, _ = cpu_icp_rate(pool, cores, cores, tar, src)
            pairs = int(min(512, max(cores, rate * budget_s)))
            times = []
            for i in range(warmup + steps):
                r, dt, _ = cpu_icp_rate(pool, cores, pairs, tar, src)
                if i >= warmup:
                    times.append(dt)
            per_step = sum(times) / len(times)
            value = pairs / per_step
            metric, unit = "icp_scan_pairs_per_s", "pairs/s"
            sample = "%d cfg-2 pairs x %d beams per step, literal Python port over %d processes" % (
                pairs, ICP_BEAMS, cores)
            config = {"workload": "cfg2 W9 LiDAR-odometry ICP, 360-beam consecutive scan pairs",
                      "pairs_per_step": pairs, "beams": ICP_BEAMS}
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# =============================================================================== GPU arm

def time_host_calls(fn, calls, bdist, torch, min_warm_calls=3, min_warm_s=0.05, lockstep=False):
    """Wall-clock seconds of `calls` back-to-back host-API calls (max over ranks).  The pinned buffers of the e2e legs
    are set up right before them, tens of ms during which the GPU idles and drops its clocks; the untimed calls
    (at least min_warm_calls and min_warm_s of them) bring it back before the timed region starts.  lockstep: the
    call contains collectives, so every rank must make the same number of calls (a fixed 6)."""
    t0 = time.perf_counter()
    n = 0
    while (n < 6) if lockstep else (n < min_warm_calls or time.perf_counter() - t0 < min_warm_s):
        fn()
        n += 1
    bdist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    torch.cuda.synchronize()
    dt = bdist.max_over_ranks(time.perf_counter() - t0)
    bdist.barrier()
    return dt


def time_host_stream(submit, calls, bdist, torch, depth=2):
    """Wall-clock seconds of `calls` steps through a submit / wait API with `depth` steps in flight: step k + 1 is
    submitted before step k's result is waited for, so its upload overlaps the read-back of step k (every step's inputs
    still cross PCIe inside the timed region, and every step's result is read back and waited for).  Max over ranks.
    Every rank makes the same number of calls (the steps rendezvous through flags)."""
    def run(n):
        pending = []
        for _ in range(n):
            pending.append(submit())
            if len(pending) >= depth:
                pending.pop(0).wait()
        for t in pending:
            t.wait()
    run(6)
    bdist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run(calls)
    torch.cuda.synchronize()
    dt = bdist.max_over_ranks(time.perf_counter() - t0)
    bdist.barrier()
    return dt


def pinned(arr):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t, t.numpy()


def bench_grid(args, rank, world, torch, devapi, bdist, synth):
    import b2slam
    G, N, K = GRID_CELLS, GRID_BEAMS, args.scans
    S, Hx, Hy = devapi.grid_scale(G, G, GRID_RESO)
    host = synth.grid_scans(12001 + rank, K, N)
    ox, oy, cx, cy = (torch.from_numpy(a).cuda() for a in host)
    hit, miss = devapi.new_planes(G, G)
    ws = devapi.new_workspace(G, G)
    pmap = torch.empty((G, G), dtype=torch.int8, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    p2p = bdist.ShardedMappingP2P(G, G, GRID_RESO) if (world > 1 and args.merge == "p2p") else None

    def step(ev=None):
        if p2p is not None:  # ray-cast, then ONE peer-memory kernel: reduce-scatter + finalize + all-gather
            p2p.update_device(ox, oy, cx, cy, events=ev)
            return
        hit.zero_()
        miss.zero_()
        if ev:
            ev[0].record()
        devapi.grid_raycast(hit, miss, S, Hx, Hy, ox, oy, cx, cy, workspace=ws)
        if ev:
            ev[1].record()
        bdist.allreduce_counts(hit, miss)
        devapi.grid_finalize(hit, miss, pmap=pmap)

    for _ in range(args.warmup):
        step()
        flush.zero_()
    torch.cuda.synchronize()
    # algorithmic bytes of one ray-cast launch: endpoints + poses + 8 B per in-grid cell visit
    hit.zero_(); miss.zero_()
    devapi.grid_raycast(hit, miss, S, Hx, Hy, ox, oy, cx, cy, workspace=ws)
    visits = int(hit.sum(dtype=torch.int64).item() + miss.sum(dtype=torch.int64).item())
    algo_bytes = 8 * K + 8 * K * N + 8 * visits

    sampler = ClockSampler(torch.cuda.current_device())
    bdist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    step_ms, ray_ms = [], []
    for _ in range(args.steps):
        e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_a.record()
        step((k0, k1))
        e_b.record()
        flush.zero_()  # evict the planes / endpoints from L2 between timed steps (not timed)
        e_b.synchronize()
        step_ms.append(e_a.elapsed_time(e_b))
        ray_ms.append(k0.elapsed_time(k1))
    torch.cuda.synchronize()
    bdist.barrier()
    clocks = sampler.stop()
    total_ms = bdist.max_over_ranks(sum(step_ms))
    ray_avg_ms = sum(ray_ms) / len(ray_ms)
    if args.dump_outputs and rank == 0:
        if p2p is not None:
            keep_grid_outputs(args, "grid", {"pmap": p2p.pmap_dev}, seed=1)
        else:
            keep_grid_outputs(args, "grid", {"hit": hit, "miss": miss, "pmap": pmap}, seed=1)

    # ---- end to end through the host-buffer API (pinned host arrays in, occupancy map out)
    e2e_steps = max(3, min(args.steps, 10))
    keep = [pinned(a) for a in host]
    h_ox, h_oy, h_cx, h_cy = (k[1] for k in keep)
    if world == 1:
        m = b2slam.Mapping(G, G, GRID_RESO)

        def e2e_step():
            m.reset()
            m.update_batch(h_ox, h_oy, h_cx, h_cy, want_pmap=True)
    else:
        sm = p2p if p2p is not None else bdist.ShardedMapping(G, G, GRID_RESO)

        def e2e_step():
            sm.update_batch(h_ox, h_oy, h_cx, h_cy)
    e2e_s = time_host_calls(e2e_step, e2e_steps, bdist, torch, lockstep=world > 1)

    # ---- the same scans in raw form (ranges + poses) through the fused-ingestion call: half the H2D bytes
    fused = None
    if world == 1 or p2p is not None:
        import math
        ranges, poses = synth.grid_scan_ranges(12001 + rank, K, N)
        keep_r, h_ranges = pinned(ranges)
        if world == 1:
            def fused_step():
                m.reset()
                m.update_scans(h_ranges, poses, -math.pi, math.pi)
            api = "Mapping.update_scans (b2s_mapping_update_scans)"
        else:
            def fused_step():
                p2p.update_scans(keep_r, poses, -math.pi, math.pi)
            api = "dist.ShardedMappingP2P.update_scans"
        fs = time_host_calls(fused_step, e2e_steps, bdist, torch, lockstep=world > 1)
        fused = {"value": world * K * N * e2e_steps / fs, "unit": "beams/s", "h2d_bytes_per_step": 4 * K * N + 32 * K,
                 "d2h_bytes_per_step": G * G, "api": api, "ms_per_step": fs / e2e_steps * 1e3}
        # the same steps through the streaming form of the call: submit step k + 1, then wait for step k
        stream_steps = max(10, min(args.steps, 40))
        if world == 1:
            # one GPU: the C-ABI host-buffer call itself (b2s_mapping_submit_scans / b2s_mapping_wait); every step clears
            # the counts first, like the device-timed step
            ss = time_host_stream(lambda: m.submit_scans(h_ranges, poses, -math.pi, math.pi, zero_first=True),
                                  stream_steps, bdist, torch)
            sapi = ("Mapping.submit_scans + MapTicket.wait (b2s_mapping_submit_scans / b2s_mapping_wait), two steps in "
                    "flight: raw ranges + poses in, int8 map out, every step")
        else:
            ss = time_host_stream(lambda: p2p.submit_scans(keep_r, poses, -math.pi, math.pi), stream_steps, bdist, torch)
            sapi = ("dist.ShardedMappingP2P.submit_scans + Ticket.wait, two steps in flight: raw ranges + poses in, merged "
                    "int8 map out, every step and rank")
        streamed = {"value": world * K * N * stream_steps / ss, "unit": "beams/s", "h2d_bytes_per_step": 4 * K * N + 24 * K,
                    "d2h_bytes_per_step": G * G, "ms_per_step": ss / stream_steps * 1e3, "api": sapi}

    peak, peak_src = measured_peaks()
    achieved = algo_bytes / (ray_avg_ms * 1e-3) / 1e9
    # DRAM bytes per launch: from the committed ncu capture of this exact workload IF the kernel source is still the
    # one that was profiled (ncu_stamp), else null
    stamp = ncu_stamp("grid_raycast")
    traffic = None
    if stamp and stamp.get("scans") == K and G == 4096 and N == 1080:
        traffic = stamp["dram_bytes_per_launch"]
    merge = merge_check(world, rank, torch, devapi, bdist, synth) if p2p is not None else None
    if p2p is not None:
        p2p.close()
    res = {
        "metric": "grid_beam_updates_per_s", "unit": "beams/s",
        "value": world * K * N * args.steps / (total_ms * 1e-3),
        "ms_per_step": total_ms / args.steps,
        "config": {"workload": "cfg3 W12 occupancy grid 4096x4096 @ 0.05 m, 1080-beam scans, known poses",
                   "scans_per_gpu_per_step": K, "beams": N, "grid": [G, G], "xyreso": GRID_RESO,
                   "hit_weight": 20.0, "cell_visits_per_step_per_gpu": visits,
                   "l2": "working set %.0f MB per step > L2 and a 256 MB buffer is rewritten between timed steps"
                         % ((2 * G * G * 4 + 8 * K * N) / 1e6),
                   "parallelism": ("single GPU" if world == 1 else
                                   "scan streams sharded by rank; count deltas merged by one peer-memory kernel "
                                   "(reduce-scatter + finalize + all-gather over NVLink)" if p2p is not None else
                                   "scan streams sharded by rank, int32 count deltas all-reduced (NCCL)")},
        "dtype": "int32 counts (f64 cell / error arithmetic)",
        "roofline": {"bound": "hbm", "kernel": "grid_raycast (+ fold of the transposed scratch plane)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic,
                     "traffic_unit": "DRAM bytes per launch (ncu --set full, profiles/r2/ncu_stamps.json; null when the kernel source changed since the capture)",
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": ray_avg_ms,
                     "cell_visits_per_s": visits / (ray_avg_ms * 1e-3)},
        "e2e": {"value": world * K * N * e2e_steps / e2e_s, "unit": "beams/s",
                "h2d_bytes_per_step": 8 * K * N + 8 * K, "d2h_bytes_per_step": G * G,
                "api": ("Mapping.update_batch (b2s_mapping_update)" if world == 1 else
                        "dist.ShardedMappingP2P.update_batch" if p2p is not None else "dist.ShardedMapping.update_batch"),
                "ms_per_step": e2e_s / e2e_steps * 1e3},
        # own kernels per step: ray-cast + fold + finalize on one GPU; clear-dirty + ray-cast + fold + publish + merge +
        # wait with the flag-synchronised peer-memory merge
        "gpu_launches": (6 if p2p is not None else 3) * args.steps,
        "clocks": clocks,
    }
    if fused:
        # headline end-to-end path: the streaming call on raw scans (4 B per beam over PCIe, the read-back of one step
        # under the upload of the next).  The blocking calls are kept beside it.
        res["e2e_blocking_call"] = res["e2e"]
        res["e2e_fused_ingestion"] = fused
        res["e2e"] = streamed
    if merge is not None:
        res["merge_bit_identical"] = merge["identical"]
        res["merge_check"] = merge
    return res


def merge_check(world, rank, torch, devapi, bdist, synth, scans=256, steps=2):
    """Driver-visible multi-GPU correctness (the reference is one process, so 'bit-identical to one GPU' is the
    contract): `steps` steps of `scans` scans per rank through the peer-memory merge, then EVERY rank ray-casts all
    ranks' scans in a single pass by itself and compares its copy of the merged occupancy map and its shard of the
    merged counts byte for byte.  The verdicts are AND-reduced over the ranks."""
    import torch.distributed as dist
    G, N = GRID_CELLS, GRID_BEAMS
    p2p = bdist.ShardedMappingP2P(G, G, GRID_RESO)
    dev = [torch.from_numpy(a).cuda() for a in synth.grid_scans(22001 + rank, scans, N)]
    for _ in range(steps):
        p2p.update_device(*dev)
    p2p.check()
    everyone = []
    for t in dev:
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        everyone.append(torch.cat(parts))
    S, Hx, Hy = devapi.grid_scale(G, G, GRID_RESO)
    hit, miss = devapi.new_planes(G, G)
    ws = devapi.new_workspace(G, G)
    for _ in range(steps):
        devapi.grid_raycast(hit, miss, S, Hx, Hy, *everyone, workspace=ws)
    pm = torch.empty((G, G), dtype=torch.int8, device="cuda")
    devapi.grid_finalize(hit, miss, pmap=pm)
    torch.cuda.synchronize()
    same_map = bool(torch.equal(pm, p2p.pmap_dev))
    n = (p2p.tile_hi - p2p.tile_lo) * 4096
    tiles = lambda plane: plane.view(G // 64, 64, G // 64, 64).permute(0, 2, 1, 3).reshape(-1)[p2p.tile_lo * 4096:p2p.tile_hi * 4096]
    same_counts = bool(torch.equal(tiles(hit), p2p.g_hit[:n]) and torch.equal(tiles(miss), p2p.g_miss[:n]))
    flag = torch.tensor([int(same_map), int(same_counts)], dtype=torch.int32, device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out = {"identical": bool(flag.min().item() == 1), "map_identical_on_every_rank": bool(flag[0].item() == 1),
           "count_shards_identical": bool(flag[1].item() == 1), "cells": G * G, "scans_per_rank": scans, "steps": steps,
           "ranks": world, "occupied_cells": int((pm == 100).sum().item()),
           "against": "one ray-cast pass over all ranks' scans, done by every rank on its own GPU"}
    p2p.close()
    return out


def bench_icp(args, rank, world, torch, devapi, bdist, synth):
    import b2slam
    xy, _ = synth.room_sequence(9001 + rank, args.icp_scans, ICP_BEAMS)
    P = xy.shape[0] - 1
    tar = torch.from_numpy(np.ascontiguousarray(xy[:-1])).cuda()
    src = torch.from_numpy(np.ascontiguousarray(xy[1:])).cuda()
    T = torch.empty((P, 3, 3), dtype=torch.float64, device="cuda")
    iters = torch.empty(P, dtype=torch.int32, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(args.warmup):
        devapi.icp_batch(tar, src, 30, 1e-3, T, iters)
        flush.zero_()
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device())
    bdist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    step_ms = []
    for _ in range(args.steps):
        e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_a.record()
        devapi.icp_batch(tar, src, 30, 1e-3, T, iters)
        e_b.record()
        flush.zero_()
        e_b.synchronize()
        step_ms.append(e_a.elapsed_time(e_b))
    torch.cuda.synchronize()
    bdist.barrier()
    clocks = sampler.stop()
    total_ms = bdist.max_over_ranks(sum(step_ms))
    if args.dump_outputs and rank == 0:
        keep_output(args, "icp_T", T)
        keep_output(args, "icp_iters", iters)
    it_total = int(iters.sum(dtype=torch.int64).item())
    evals = it_total * ICP_BEAMS * ICP_BEAMS
    flops = it_total * (5 * ICP_BEAMS * ICP_BEAMS + 24 * ICP_BEAMS) + P * 16 * ICP_BEAMS
    step_s = sum(step_ms) / len(step_ms) * 1e-3
    hbm_bytes = P * (8 * (ICP_BEAMS + ICP_BEAMS) + 72 + 4)

    # ---- end to end through the host-buffer API: the scan stream in pinned host memory, T and iteration counts out.
    # cfg 2 IS a sequence (pair k = scans k, k+1), so the call a user makes is process_sequence (each scan crosses
    # PCIe once); the pair form process_batch(scans[:-1], scans[1:]) is timed beside it.
    e2e_steps = max(3, min(args.steps, 10))
    icp = b2slam.ICP()
    keep_q, h_seq = pinned(xy)
    e2e_s = time_host_calls(lambda: icp.process_sequence(h_seq), e2e_steps, bdist, torch)
    keep_t, h_tar = pinned(xy[:-1])
    keep_s, h_src = pinned(xy[1:])
    pair_s = time_host_calls(lambda: icp.process_batch(h_tar, h_src), e2e_steps, bdist, torch)
    # the same stream as raw ranges (what the sensor delivers): laserToNumpy runs inside the kernel, 4 B per beam
    import math
    keep_r, h_rng = pinned(np.hypot(xy[:, 0, :], xy[:, 1, :]).astype(np.float32))
    raw_s = time_host_calls(lambda: icp.process_scans(h_rng, -math.pi, math.pi), e2e_steps, bdist, torch)
    # streaming form of the sequence call: submit stream k + 1, then wait for stream k (two in flight)
    stream_steps = max(10, min(args.steps, 40))
    seq_stream_s = time_host_stream(lambda: icp.submit_sequence(h_seq), stream_steps, bdist, torch)
    # ... and of the raw-range call: half the bytes per scan, which is what counts once several ranks share the host
    raw_stream_s = time_host_stream(lambda: icp.submit_scans(h_rng, -math.pi, math.pi), stream_steps, bdist, torch)

    peak, peak_src = measured_peaks()
    import ctypes
    from b2slam import _lib
    fp64_peak = ctypes.c_double(0.0)
    _lib.check(_lib.lib().b2s_measure_fp64_peak(ctypes.byref(fp64_peak)))
    return {
        "metric": "icp_scan_pairs_per_s", "unit": "pairs/s",
        "value": world * P * args.steps / (total_ms * 1e-3), "ms_per_step": total_ms / args.steps,
        "config": {"workload": "cfg2 W9 LiDAR-odometry ICP, 10k-scan 360-beam room sequence, consecutive pairs",
                   "pairs_per_gpu_per_step": P, "beams": ICP_BEAMS, "max_iter": 30, "tolerance": 1e-3,
                   "mean_iterations": it_total / P,
                   "l2": "a 256 MB buffer is rewritten between timed steps",
                   "parallelism": "independent pairs sharded by rank, no collective" if world > 1 else "single GPU"},
        "dtype": "f64",
        "roofline": {"bound": "hbm", "kernel": "icp_batch_kernel", "achieved": hbm_bytes / step_s / 1e9, "peak": peak,
                     "unit": "GB/s", "frac": hbm_bytes / step_s / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                     "note": "compute (FP64 issue) bound by design: each pair reads 8(N+M)+76 B once and iterates on chip, "
                             "so the HBM fraction is expected to be << 1%",
                     "nn_search": "exact, warp-level + per-lane block pruning, surviving (point, block) pairs queued and spread over the lanes (identical correspondences to the N x M brute force)",
                     "brute_force_equivalent_pair_evals_per_s": evals / step_s,
                     "brute_force_equivalent_fp64_tflops": flops / step_s / 1e12,
                     "fp64_peak_tflops_nominal": FP64_PEAK_TFLOPS,
                     "fp64_peak_tflops_measured_same_run": fp64_peak.value,
                     "fp64_pipe_executed": (lambda st: None if not st else {k: st[k] for k in st if k not in ("sources", "sha1")})(ncu_stamp("icp_360")),
                     "fp64_note": "the pruned search executes a fraction of the brute-force evaluations, so the brute-force-"
                                  "equivalent rate is not a utilisation; fp64_pipe_executed is: the share of the FP64 pipe and "
                                  "the executed warp instructions of this kernel from the committed ncu capture "
                                  "(profiles/r2/ncu_stamps.json, null when the kernel source changed since)"},
        "e2e": {"value": world * P * stream_steps / raw_stream_s, "unit": "pairs/s",
                "h2d_bytes_per_step": int(h_rng.nbytes), "d2h_bytes_per_step": P * 76,
                "api": "ICP.submit_scans + IcpTicket.wait (b2s_icp_submit_scans / b2s_icp_wait), two streams in flight: raw "
                       "ranges in (what the sensor delivers; laserToNumpy inside the kernel), T and iteration counts out",
                "ms_per_step": raw_stream_s / stream_steps * 1e3},
        "e2e_streaming_sequence": {"value": world * P * stream_steps / seq_stream_s, "unit": "pairs/s",
                                   "h2d_bytes_per_step": int(h_seq.nbytes), "d2h_bytes_per_step": P * 76,
                                   "api": "ICP.submit_sequence + IcpTicket.wait (b2s_icp_submit_sequence / b2s_icp_wait), "
                                          "two streams in flight, float32 points in (PCIe-bound: 28.8 MB per stream)",
                                   "ms_per_step": seq_stream_s / stream_steps * 1e3},
        "e2e_blocking_call": {"value": world * P * e2e_steps / e2e_s, "unit": "pairs/s",
                              "h2d_bytes_per_step": int(h_seq.nbytes), "d2h_bytes_per_step": P * 76,
                              "api": "ICP.process_sequence (b2s_icp_process_sequence)", "ms_per_step": e2e_s / e2e_steps * 1e3},
        "e2e_pair_form": {"value": world * P * e2e_steps / pair_s, "unit": "pairs/s",
                          "h2d_bytes_per_step": int(h_tar.nbytes + h_src.nbytes), "d2h_bytes_per_step": P * 76,
                          "api": "ICP.process_batch (b2s_icp_process)", "ms_per_step": pair_s / e2e_steps * 1e3},
        "e2e_fused_ingestion": {"value": world * P * e2e_steps / raw_s, "unit": "pairs/s",
                                "h2d_bytes_per_step": int(h_rng.nbytes), "d2h_bytes_per_step": P * 76,
                                "api": "ICP.process_scans (b2s_icp_process_scans)", "ms_per_step": raw_s / e2e_steps * 1e3},
        "gpu_launches": args.steps,
        "clocks": clocks,
    }


def device_pairs(torch, seed, pairs, beams, chunk=65536):
    """cfg 4 input: the synth.icp_pairs formulae evaluated with torch on the GPU (float32 points; 17.3 GB for 10^6 pairs
    would not be worth generating on the host)."""
    import math
    g = torch.Generator(device="cuda").manual_seed(seed)
    tar = torch.empty((pairs, 2, beams), dtype=torch.float32, device="cuda")
    src = torch.empty_like(tar)
    phi = torch.linspace(-math.pi, math.pi, beams, dtype=torch.float64, device="cuda")[None, :]
    for s in range(0, pairs, chunk):
        e = min(pairs, s + chunk)
        n = e - s
        u = lambda lo, hi, shape: lo + (hi - lo) * torch.rand(shape, generator=g, dtype=torch.float64, device="cuda")
        r0, amp, psi = u(3, 8, (n, 1)), u(0.5, 2, (n, 1)), u(0, 2 * math.pi, (n, 1))
        k = torch.randint(2, 6, (n, 1), generator=g, device="cuda").double()
        base = r0 + amp * torch.sin(k * phi + psi)
        noise = lambda: torch.randn((n, beams), generator=g, dtype=torch.float64, device="cuda") * 0.01
        rt = (base + noise()).clamp(0.10, 30.0)
        rs = (base + noise()).clamp(0.10, 30.0)
        tx, ty, th = u(-0.15, 0.15, (n, 1)), u(-0.15, 0.15, (n, 1)), u(-0.08, 0.08, (n, 1))
        tar[s:e, 0], tar[s:e, 1] = (rt * torch.cos(phi)).float(), (rt * torch.sin(phi)).float()
        sx, sy = rs * torch.cos(phi), rs * torch.sin(phi)
        c, sn = torch.cos(th), torch.sin(th)
        src[s:e, 0], src[s:e, 1] = (c * sx - sn * sy + tx).float(), (sn * sx + c * sy + ty).float()
    return tar, src


def bench_cfg4(args, rank, world, torch, devapi, bdist):
    """BASELINE.json config 4: 10^6 independent 1080-beam ICP pairs sharded over the ranks (strong scaling, no
    collective).  Parity: the first 64 pairs of every rank against oracle.c (T to 1e-9, identical iteration counts)."""
    import torch.distributed as dist
    total, beams = args.cfg4_pairs, 1080
    lo, hi = bdist.shard_bounds(total, rank, world)
    tar, src = device_pairs(torch, 4001 + rank, hi - lo, beams)
    T = torch.empty((hi - lo, 3, 3), dtype=torch.float64, device="cuda")
    it = torch.empty(hi - lo, dtype=torch.int32, device="cuda")
    devapi.icp_batch(tar[:8192], src[:8192], 30, 1e-3)
    torch.cuda.synchronize()
    times = []
    for _ in range(2):
        bdist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        devapi.icp_batch(tar, src, 30, 1e-3, T, it)
        b.record()
        torch.cuda.synchronize()
        times.append(bdist.max_over_ranks(a.elapsed_time(b)))
    ms = min(times)
    if args.dump_outputs and rank == 0:
        idx = seeded_sample(hi - lo, DUMP_PAIRS, seed=2)
        args.outputs["cfg4_pairs"] = idx.astype(np.float64)
        idx = torch.from_numpy(idx).cuda()
        keep_output(args, "cfg4_T", T[idx])
        keep_output(args, "cfg4_iters", it[idx])
    from oracle import corc                     # the checker, on a sample; never the thing timed
    sample = min(64, hi - lo)
    want_T, want_it = corc.icp_batch(tar[:sample].cpu().numpy(), src[:sample].cpu().numpy(), 30, 1e-3)
    got_T, got_it = T[:sample].cpu().numpy(), it[:sample].cpu().numpy()
    ok = bool(np.array_equal(got_it, want_it) and np.abs(got_T - want_T).max() < 1e-9)
    flag = torch.tensor([int(ok)], dtype=torch.int32, device="cuda")
    iters = it.sum(dtype=torch.int64).reshape(1).clone()
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        dist.all_reduce(iters)
    fp64 = ncu_stamp("icp_1080")
    return {"workload": "cfg4: %d independent 1080-beam ICP pairs sharded over the ranks, max_iter 30, tolerance 1e-3" % total,
            "value": total / (ms * 1e-3), "unit": "pairs/s", "ms": ms, "n_gpus": world, "scaling": "strong",
            "pairs_per_gpu": hi - lo, "mean_iterations": float(iters.item()) / total,
            "parity": {"ok": bool(flag.item() == 1), "pairs_per_rank": sample, "against": "oracle.c (float64)",
                       "tolerance": "T 1e-9 abs, iteration counts identical"},
            "fp64_pipe": None if not fp64 else {k: fp64[k] for k in fp64 if k not in ("sources", "sha1")}}


def bench_cfg5(args, rank, world, torch, devapi, bdist, synth):
    """BASELINE.json config 5: one global 16384 x 16384 grid from 8 scan streams; the streams are split over the ranks
    (strong scaling) and the int32 count deltas merged over peer memory.  Parity: every rank also ray-casts all 8
    streams alone and compares the merged occupancy map and its shard of the merged counts byte for byte."""
    import torch.distributed as dist
    G, streams, K, N = 16384, 8, args.cfg5_scans, GRID_BEAMS
    lo, hi = bdist.shard_bounds(streams, rank, world)
    gen = lambda s: synth.grid_scans(5001 + s, K, N, half_extent_m=380.0)
    mine = [gen(s) for s in range(lo, hi)]
    dev = [torch.from_numpy(np.concatenate([p[k] for p in mine])).cuda() for k in range(4)] if mine else None
    sm = bdist.ShardedMappingP2P(G, G, GRID_RESO)
    empty = [torch.empty((0, N), dtype=torch.float32, device="cuda"), torch.empty((0, N), dtype=torch.float32, device="cuda"),
             torch.empty(0, dtype=torch.float32, device="cuda"), torch.empty(0, dtype=torch.float32, device="cuda")]
    batch = dev if dev is not None else empty
    sm.update_device(*batch)
    torch.cuda.synchronize()
    bdist.barrier()
    reps = 5
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        sm.update_device(*batch)
    b.record()
    torch.cuda.synchronize()
    sm.check()
    if args.dump_outputs and rank == 0:
        keep_grid_outputs(args, "cfg5", {"pmap": sm.pmap_dev}, seed=3)
    ms = bdist.max_over_ranks(a.elapsed_time(b)) / reps
    # parity: all 8 streams in one pass on this GPU, (1 + reps) times like the merged object saw them
    S, Hx, Hy = devapi.grid_scale(G, G, GRID_RESO)
    hit, miss = devapi.new_planes(G, G)
    ws = devapi.new_workspace(G, G)
    for s in range(streams):
        one = [torch.from_numpy(a_).cuda() for a_ in (mine[s - lo] if lo <= s < hi else gen(s))]
        for _ in range(1 + reps):
            devapi.grid_raycast(hit, miss, S, Hx, Hy, *one, workspace=ws)
        del one
    pm = torch.empty((G, G), dtype=torch.int8, device="cuda")
    devapi.grid_finalize(hit, miss, pmap=pm)
    torch.cuda.synchronize()
    n = (sm.tile_hi - sm.tile_lo) * 4096
    tiles = lambda plane: plane.view(G // 64, 64, G // 64, 64).permute(0, 2, 1, 3).reshape(-1)[sm.tile_lo * 4096:sm.tile_hi * 4096]
    ok = bool(torch.equal(pm, sm.pmap_dev) and torch.equal(tiles(hit), sm.g_hit[:n]) and torch.equal(tiles(miss), sm.g_miss[:n]))
    flag = torch.tensor([int(ok)], dtype=torch.int32, device="cuda")
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out = {"workload": "cfg5: global 16384x16384 grid @ 0.05 m from 8 scan streams x %d scans x %d beams, streams split over "
                       "the ranks, count deltas merged over NVLink peer memory" % (K, N),
           "value": streams * K * N / (ms * 1e-3), "unit": "beams/s", "ms_per_step": ms, "n_gpus": world, "scaling": "strong",
           "streams_per_gpu": hi - lo, "occupied_cells": int((pm == 100).sum().item()),
           "counts_checksum": int(hit.sum(dtype=torch.int64).item() * 1000003 + miss.sum(dtype=torch.int64).item()),
           "parity": {"ok": bool(flag.item() == 1), "against": "one single-GPU ray-cast pass over all 8 streams, done by every rank",
                      "compared": "int8 occupancy map on every rank + each rank's shard of the int32 counts, byte for byte"}}
    sm.close()
    return out


def drop_in_latency(torch, synth):
    """Single-call latency of the reference-signature methods (what a ROS node sees per scan)."""
    import b2slam
    out = {}
    tar, src, _ = synth.icp_pairs(7001, 1, 360)                       # cfg 1: the W7 pair
    t3, s3 = synth.homogeneous(tar[0].astype(np.float64)), synth.homogeneous(src[0].astype(np.float64))
    icp = b2slam.ICP(max_iter=10, tolerance=0.0)                      # W7 icp.launch:10-11
    for _ in range(5):
        icp.process(t3, s3)
    t0 = time.perf_counter()
    for _ in range(50):
        icp.process(t3, s3)
    out["ICP.process cfg1 (360 beams, max_iter 10, tolerance 0) ms"] = (time.perf_counter() - t0) / 50 * 1e3
    from b2slam import _lib
    _lib.check(_lib.lib().b2s_tune(b"icp_graph", 0))                  # the same call as plain stream operations
    for _ in range(5):
        icp.process(t3, s3)
    t0 = time.perf_counter()
    for _ in range(50):
        icp.process(t3, s3)
    out["ICP.process cfg1 without the captured CUDA graph ms"] = (time.perf_counter() - t0) / 50 * 1e3
    _lib.check(_lib.lib().b2s_tune(b"icp_graph", 1))
    ox, oy, cx, cy = synth.grid_scans(12001, 64, 1080, half_extent_m=8.0)
    for shape, reso in (((200, 200), 0.1), ((4096, 4096), 0.05)):
        m = b2slam.Mapping(shape[0], shape[1], reso)
        for k in range(4):
            m.update(ox[k].astype(np.float64), oy[k].astype(np.float64), float(cx[k]), float(cy[k]))
        t0 = time.perf_counter()
        for k in range(4, 36):
            m.update(ox[k].astype(np.float64), oy[k].astype(np.float64), float(cx[k]), float(cy[k]))
        out["Mapping.update one 1080-beam scan, %dx%d map (float64 pmap returned) ms" % shape] = \
            (time.perf_counter() - t0) / 32 * 1e3
        t0 = time.perf_counter()
        for k in range(36, 64):
            m.update_batch(ox[k:k + 1], oy[k:k + 1], cx[k:k + 1], cy[k:k + 1], want_pmap=False)
        out["Mapping.update_batch one scan, %dx%d map (no map read-back) ms" % shape] = \
            (time.perf_counter() - t0) / 28 * 1e3
    torch.cuda.synchronize()
    return out


def cpu_baselines(args, synth):
    cores = host_cores()
    ctx = mp.get_context("fork")
    out = {}
    with ctx.Pool(cores) as pool:
        scans = 256 * cores   # ~10 s of wall time on all cores (the literal port does ~30 k beams/s per core)
        data = synth.grid_scans(12001, scans, GRID_BEAMS)
        rate, dt, _ = cpu_grid_rate(pool, cores, scans, data)
        out["grid"] = {"value": rate, "unit": "beams/s", "cores": cores, "kind": "port",
                       "sample": "first %d cfg-3 scans x %d beams, literal Python port (oracle/pyref.py) over %d "
                                 "processes, %.1f s wall" % (scans, GRID_BEAMS, cores, dt)}
        pairs = 8 * cores     # ~15 s of wall time on all cores (~0.6 pairs/s per core at 360 beams)
        xy, _ = synth.room_sequence(9001, 513, ICP_BEAMS)
        rate, dt, _ = cpu_icp_rate(pool, cores, pairs, xy[:-1], xy[1:])
        out["icp"] = {"value": rate, "unit": "pairs/s", "cores": cores, "kind": "port",
                      "sample": "%d evenly spaced cfg-2 pairs x %d beams, literal Python port (oracle/pyref.py) over %d "
                                "processes, %.1f s wall" % (pairs, ICP_BEAMS, cores, dt)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="timed steps (100 x 2.5 ms: a quarter-second timed region)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2slam", choices=["b2slam", "reference"])
    ap.add_argument("--workload", default="grid", choices=["grid", "icp"])
    ap.add_argument("--scans", type=int, default=16384, help="grid scans per GPU per step")
    ap.add_argument("--icp-scans", type=int, default=ICP_SCANS)
    ap.add_argument("--grid-variant", type=int, default=0)
    ap.add_argument("--icp-r", type=int, default=0, help="force ICP source points per thread (tuning)")
    ap.add_argument("--icp-prune", type=int, default=-1, help="0: brute-force NN, 1: per-lane block pruning, 2: warp-level + per-lane, 3: warp-level only, 4: queued (default) (tuning)")
    ap.add_argument("--merge", default="p2p", choices=["p2p", "nccl"], help="multi-GPU grid merge")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", default="both", choices=["both", "primary"])
    ap.add_argument("--cfg4-pairs", type=int, default=1000000, help="BASELINE.json config 4: total ICP pairs (0 skips it)")
    ap.add_argument("--cfg5-scans", type=int, default=4096, help="BASELINE.json config 5: scans per stream (0 skips it)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b2slam arm")
    args.outputs = {}
    args.warmup = max(args.warmup, 3) if args.impl == "b2slam" else args.warmup

    if args.impl == "reference":
        return run_reference(args)

    # keep stdout to the one JSON line: whatever the libraries print (NCCL's version banner, warnings) goes to
    # stderr -- at the file-descriptor level, since NCCL writes from C -- until the line itself is printed
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    from b2slam import _lib, devapi, synth
    from b2slam import dist as bdist
    if not torch.cuda.is_available() or _lib.device_count() <= 0:
        raise SystemExit("bench.py needs a CUDA device: b2slam has no CPU fallback")
    rank, local_rank, world = bdist.init()
    if args.grid_variant:
        _lib.check(_lib.lib().b2s_tune(b"grid_variant", args.grid_variant))
    if args.icp_prune >= 0:
        _lib.check(_lib.lib().b2s_tune(b"icp_prune", args.icp_prune))
    if args.icp_r:
        _lib.check(_lib.lib().b2s_tune(b"icp_src_per_thread", args.icp_r))

    results = {}
    order = ["grid", "icp"] if args.workload == "grid" else ["icp", "grid"]
    if args.only == "primary":
        order = order[:1]
    for name in order:
        fn = bench_grid if name == "grid" else bench_icp
        results[name] = fn(args, rank, world, torch, devapi, bdist, synth)
        torch.cuda.synchronize()
        bdist.barrier()

    extra = {}
    if args.only == "both":
        if args.cfg4_pairs > 0:
            extra["cfg4"] = bench_cfg4(args, rank, world, torch, devapi, bdist)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            bdist.barrier()
        if args.cfg5_scans > 0:
            extra["cfg5"] = bench_cfg5(args, rank, world, torch, devapi, bdist, synth)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            bdist.barrier()

    cpu = {}
    latency = None
    if rank == 0 and world == 1 and args.only == "both":
        latency = drop_in_latency(torch, synth)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baselines(args, synth)
    bdist.barrier()

    if rank == 0:
        prim = results[order[0]]
        line = {
            "metric": prim["metric"], "value": prim["value"], "unit": prim["unit"], "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": prim["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": prim["dtype"],
            "data": "synthetic", "config": prim["config"], "roofline": prim["roofline"], "e2e": prim["e2e"],
            **{k: prim[k] for k in ("e2e_blocking_call", "e2e_fused_ingestion", "e2e_pair_form", "e2e_streaming_sequence", "merge_bit_identical",
                                    "merge_check") if k in prim},
            "gpu_launches": sum(r["gpu_launches"] for r in results.values()), "clocks": prim["clocks"],
            "cpu_baseline": cpu.get(order[0]),
        }
        line.update(extra)
        if latency:
            line["drop_in_latency_ms"] = latency
        if len(order) > 1:
            sec = results[order[1]]
            sec["cpu_baseline"] = cpu.get(order[1])
            line[order[1]] = sec
        if args.dump_outputs:
            write_outputs(args.outputs, args.dump_outputs)
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
