"""Where a variant-6 ray-cast CTA spends its time: phase clocks at the bench launch (cfg 3: seed 12001, 16 384 scans x
1080 beams into 4096^2 @ 5 cm).
   python profiles/scripts/grid_phases.py OUT_DIR [layouts, default 0,1]
Builds the library with -DB2S_GRID_PHASES into OUT_DIR (the package's own libb2slam.so is not touched), then, per
tile layout, runs one warm-up and one recorded launch (planes zeroed, L2 flushed) and writes OUT_DIR/phases_layout<L>.json.
Thread 0 of every CTA stamps clock64 at start, box known, tile zeroed, march done and end; lane 0 of every warp stamps
its own march end.  Clocks are per SM, so only differences within one SM are used.  Reported, in SM cycles:
- per phase, the mean over the CTAs that take the tile, and each phase's share of all CTA cycles (fallback CTAs are
  counted whole under "fallback");
- the warp-slot efficiency of the march: sum over warps of their march cycles / (warps x the CTA's march phase); the
  rest is the idle warp-slots at the barrier after the march;
- the mean number of marching warps per SM while at least one warp of that SM marches;
- the flush share: flush cycles / all CTA cycles.
The stamps cost a few instructions per CTA and per warp; the launch time printed beside them is that of the
instrumented build."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from b2slam import _lib

CSRC = os.path.join(ROOT, "a-2d-lidar-based-slam-system-for-wheeled-mobile-robots_b200", "csrc")
V6_SCANS, V6_SECTOR, WORDS = 16, 64, 8 + 32  # csrc/b2s_grid.cu (V6_PHASE_WORDS)


def build(out):
    lib = os.path.join(out, "libb2slam.so")
    subprocess.check_call(["make", "-s", "-j8", "-C", CSRC, "BUILD=" + os.path.join(out, "obj"), "OUT=" + lib,
                           "EXTRA=-DB2S_GRID_PHASES"])
    return lib


def live_warps(sm, t0, t1):
    """Time-weighted mean number of open intervals [t0, t1) per SM, over the time at least one is open."""
    res = []
    for s in np.unique(sm):
        a, b = t0[sm == s], t1[sm == s]
        ev = np.concatenate([a, b])
        d = np.concatenate([np.ones_like(a), -np.ones_like(b)])
        o = np.argsort(ev, kind="stable")
        ev, d = ev[o], np.cumsum(d[o])
        dt = np.diff(ev).astype(np.float64)
        live = d[:-1]
        busy = dt[live > 0].sum()
        if busy > 0:
            res.append(float((dt * live).sum() / busy))
    return float(np.mean(res))


def analyse(rec, ms):
    sm, t = rec[:, 0], rec[:, 1:6].astype(np.int64)
    fell, nw = rec[:, 6] == 1, int(rec[0, 7])
    tile = ~fell
    total = t[:, 4] - t[:, 0]
    ph = {"box": t[:, 1] - t[:, 0], "zero": t[:, 2] - t[:, 1], "march": t[:, 3] - t[:, 2], "flush": t[:, 4] - t[:, 3]}
    all_cycles = float(total.sum())
    wend = rec[tile][:, 8:8 + nw].astype(np.int64)
    mstart, mdone = t[tile][:, 2:3], t[tile][:, 3:4]
    wcyc = wend - mstart
    slot_eff = float(wcyc.sum() / (nw * (mdone - mstart)).sum())
    smw = np.repeat(sm[tile], nw)
    span = {int(s): int(t[sm == s, 4].max() - t[sm == s, 0].min()) for s in np.unique(sm)}
    return {
        "launch_ms_instrumented": ms,
        "ctas": int(len(rec)), "tile_ctas": int(tile.sum()), "fallback_ctas": int(fell.sum()), "warps_per_cta": nw,
        "tile_cta_mean_cycles": {k: float(v[tile].mean()) for k, v in ph.items()} | {"total": float(total[tile].mean())},
        "fallback_cta_mean_cycles": float(total[fell].mean()) if fell.any() else None,
        "share_of_cta_cycles": {k: float(v[tile].sum() / all_cycles) for k, v in ph.items()}
                               | {"fallback": float(total[fell].sum() / all_cycles)},
        "march_warp_slot_efficiency": slot_eff,
        "march_idle_warp_slots_at_barrier": 1.0 - slot_eff,
        "march_warp_cycles_longest_over_mean": float((wcyc.max(axis=1) / wcyc.mean(axis=1)).mean()),
        "mean_marching_warps_per_sm": live_warps(smw, np.repeat(mstart[:, 0], nw), wend.reshape(-1)),
        "flush_share": float(ph["flush"][tile].sum() / all_cycles),
        "sm_span_cycles_mean": float(np.mean(list(span.values()))),
        "sms": len(span),
    }


def main():
    out = os.path.abspath(sys.argv[1])
    layouts = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "0,1").split(",")]
    os.makedirs(out, exist_ok=True)
    _lib.LIB_PATH = build(out)
    from b2slam import devapi, synth
    L = _lib.lib()
    L.b2s_grid_phases_buffer.argtypes = [ctypes.c_void_p]
    G, K, N = 4096, 16384, 1080
    S, Hx, Hy = devapi.grid_scale(G, G, 0.05)
    ox, oy, cx, cy = (torch.from_numpy(a).cuda() for a in synth.grid_scans(12001, K, N))
    ctas = ((K + V6_SCANS - 1) // V6_SCANS) * ((N + V6_SECTOR - 1) // V6_SECTOR)
    rec = torch.zeros(ctas * WORDS, dtype=torch.int64, device="cuda")
    _lib.check(L.b2s_grid_phases_buffer(ctypes.c_void_p(rec.data_ptr())))
    hit, miss = devapi.new_planes(G, G)
    ws = devapi.new_workspace(G, G)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    for lay in layouts:
        _lib.check(L.b2s_tune(b"grid_tile_layout", lay))
        for it in range(2):
            hit.zero_(); miss.zero_(); rec.zero_(); flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            devapi.grid_raycast(hit, miss, S, Hx, Hy, ox, oy, cx, cy, workspace=ws)
            b.record()
            torch.cuda.synchronize()
        r = analyse(rec.view(ctas, WORDS).cpu().numpy(), a.elapsed_time(b))
        r = {"workload": "cfg3 bench launch: %d scans x %d beams into %d^2 @ 0.05 m" % (K, N, G),
             "device": card[0] if card else None, "grid_tile_layout": lay,
             "visits": int(hit.sum(dtype=torch.int64).item() + miss.sum(dtype=torch.int64).item())} | r
        with open(os.path.join(out, "phases_layout%d.json" % lay), "w") as fh:
            json.dump(r, fh, indent=1)
        print(json.dumps(r))
    _lib.check(L.b2s_grid_phases_buffer(None))
    _lib.check(L.b2s_tune(b"grid_tile_layout", 1))


if __name__ == "__main__":
    main()
