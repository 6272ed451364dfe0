"""A/B of ray-cast variant 5 and the two tile layouts of variant 6 at the bench launch (cfg 3: seed 12001, 16 384 scans x 1080 beams, 4096^2 @ 5 cm).
   python profiles/scripts/grid_tile_ab.py [launches per variant, default 30] [scans, default 16384]
Alternates variant 5, variant 6 with grid_tile_layout 0 (1024 threads, one unit per warp) and variant 6 with layout 1
(512 threads, two units per warp) launch by launch in one process, on zeroed planes with L2 flushed before every
launch, and prints one JSON line: median / min / max ms per launch (CUDA events around ray-cast + fold), the share of
variant-6 CTAs that fall back to the variant-5 march (the kernel's rule, evaluated on the host), registers / shared
memory / resident CTAs of the kernels (cuobjdump of the built library), and whether the planes of all three are equal
byte for byte."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from b2slam import _lib, devapi, synth

V6_SCANS, V6_SECTOR, V6_TILE_WORDS = 16, 64, 27 * 1024  # csrc/b2s_grid.cu


def fallback_share(host, G, S, H):
    """Share of variant-6 CTAs whose box does not fit the tile or that hold a clipped ray (csrc/b2s_grid.cu)."""
    ox, oy, cx, cy = (a.astype(np.float64) for a in host)
    K, N = ox.shape
    hx, hy = np.trunc(S * (ox + H)).astype(np.int64), np.trunc(S * (oy + H)).astype(np.int64)
    sx, sy = np.trunc(S * (cx + H)).astype(np.int64), np.trunc(S * (cy + H)).astype(np.int64)
    sx, sy = np.broadcast_to(sx[:, None], hx.shape), np.broadcast_to(sy[:, None], hy.shape)
    live = ~((hx == sx) & (hy == sy))
    live &= ~((np.maximum(sx, hx) < 0) | (np.minimum(sx, hx) >= G) | (np.maximum(sy, hy) < 0) | (np.minimum(sy, hy) >= G))
    fell, total = 0, 0
    for s0 in range(0, K, V6_SCANS):
        for b0 in range(0, N, V6_SECTOR):
            sl = (slice(s0, s0 + V6_SCANS), slice(b0, b0 + V6_SECTOR))
            lv = live[sl]
            total += 1
            if not lv.any():
                continue
            xs = np.concatenate([sx[sl][lv], hx[sl][lv]])
            ys = np.concatenate([sy[sl][lv], hy[sl][lv]])
            clipped = xs.min() < 0 or xs.max() >= G or ys.min() < 0 or ys.max() >= G
            w, h = xs.max() - xs.min() + 1, ys.max() - ys.min() + 1
            fell += bool(clipped or w * (h | 1) > V6_TILE_WORDS)
    return fell / total


def resources():
    """Registers, static + dynamic shared memory and resident CTAs per SM of the v5 / v6 kernels (float32 input)."""
    lib = os.path.join(ROOT, "a-2d-lidar-based-slam-system-for-wheeled-mobile-robots_b200", "libb2slam.so")
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout
    res, fn = {}, None
    for line in out.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+)", line)
        if m and fn:
            if "grid_raycast_v4ILi1ELi0ELb1E" in fn:
                res["v5"] = {"regs": int(m.group(1)), "stack": int(m.group(2)), "smem_static": int(m.group(3)),
                             "threads": 256, "smem_dynamic": 0}
            elif "grid_raycast_v6ILi0ELi1E" in fn or "grid_raycast_v6ILi0ELi2E" in fn:
                units = 1 if "ILi0ELi1E" in fn else 2
                res["v6_layout%d" % (units - 1)] = {"regs": int(m.group(1)), "stack": int(m.group(2)),
                                                    "smem_static": int(m.group(3)), "threads": 1024 // units,
                                                    "smem_dynamic": V6_TILE_WORDS * 4}
    # B200 per SM: 64 K registers, 2048 threads, 228 KB shared memory, 32 CTAs (SHARED includes the 1 KB per CTA
    # that the system reserves)
    for r in res.values():
        by_regs = 65536 // (r["regs"] * r["threads"])
        by_smem = (228 * 1024) // (r["smem_static"] + r["smem_dynamic"])
        r["ctas_per_sm"] = min(by_regs, by_smem, 2048 // r["threads"], 32)
        r["occupancy"] = r["ctas_per_sm"] * r["threads"] / 2048
    return res


def main():
    launches = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    K = int(sys.argv[2]) if len(sys.argv) > 2 else 16384
    G, N = 4096, 1080
    S, Hx, Hy = devapi.grid_scale(G, G, 0.05)
    host = synth.grid_scans(12001, K, N)
    ox, oy, cx, cy = (torch.from_numpy(a).cuda() for a in host)
    arms = {"v5": (5, 1), "v6_layout0": (6, 0), "v6_layout1": (6, 1)}  # grid_variant, grid_tile_layout
    planes = {a: devapi.new_planes(G, G) for a in arms}
    ws = devapi.new_workspace(G, G)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    ms = {a: [] for a in arms}
    for it in range(3 + launches):
        for v, (variant, layout) in arms.items():
            _lib.check(_lib.lib().b2s_tune(b"grid_variant", variant))
            _lib.check(_lib.lib().b2s_tune(b"grid_tile_layout", layout))
            hit, miss = planes[v]
            hit.zero_(); miss.zero_(); flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            devapi.grid_raycast(hit, miss, S, Hx, Hy, ox, oy, cx, cy, workspace=ws)
            b.record()
            torch.cuda.synchronize()
            if it >= 3:
                ms[v].append(a.elapsed_time(b))
    _lib.check(_lib.lib().b2s_tune(b"grid_tile_layout", 1))
    (h5, m5), (h0, m0), (h6, m6) = planes["v5"], planes["v6_layout0"], planes["v6_layout1"]
    visits = int(h6.sum(dtype=torch.int64).item() + m6.sum(dtype=torch.int64).item())
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    stat = lambda x: {"median_ms": float(np.median(x)), "min_ms": float(np.min(x)), "max_ms": float(np.max(x)),
                      "launches": len(x)}
    print(json.dumps({
        "workload": "cfg3 bench launch: %d scans x %d beams into %d^2 @ 0.05 m, L2 flushed before every launch" % (K, N, G),
        "device": card[0] if card else None,
        **{a: stat(x) for a, x in ms.items()},
        "layout1_over_layout0_median": float(np.median(ms["v6_layout1"]) / np.median(ms["v6_layout0"])),
        "v5_over_layout1_median": float(np.median(ms["v5"]) / np.median(ms["v6_layout1"])),
        "v6_fallback_cta_share": fallback_share(host, G, S, Hx),
        "resources": resources(),
        "planes_byte_identical": bool(torch.equal(h5, h6) and torch.equal(m5, m6) and torch.equal(h0, h6) and
                                      torch.equal(m0, m6)),
        "visits": visits}))


if __name__ == "__main__":
    main()
