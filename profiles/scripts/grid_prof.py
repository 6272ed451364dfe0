"""Minimal grid ray-cast launcher for ncu / timing: the cfg-3 bench launch (16 384 scans x 1080 beams, 4096^2 @ 5 cm).
   python profiles/scripts/grid_prof.py [variant 1..6] [scans]
Prints the CUDA-event time of the ray-cast (+ fold) averaged over 10 launches on zeroed planes, L2 flushed between."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from b2slam import _lib, devapi, synth

variant = int(sys.argv[1]) if len(sys.argv) > 1 else 5
K = int(sys.argv[2]) if len(sys.argv) > 2 else 16384
G, N = 4096, 1080
_lib.check(_lib.lib().b2s_tune(b"grid_variant", variant))
S, Hx, Hy = devapi.grid_scale(G, G, 0.05)
ox, oy, cx, cy = (torch.from_numpy(a).cuda() for a in synth.grid_scans(12001, K, N))
hit, miss = devapi.new_planes(G, G)
ws = devapi.new_workspace(G, G)
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
ms = []
for it in range(13):
    hit.zero_(); miss.zero_(); flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    devapi.grid_raycast(hit, miss, S, Hx, Hy, ox, oy, cx, cy, workspace=ws)
    b.record()
    torch.cuda.synchronize()
    if it >= 3:
        ms.append(a.elapsed_time(b))
visits = int(hit.sum(dtype=torch.int64).item() + miss.sum(dtype=torch.int64).item())
print("variant %d scans %d: %.4f ms (min %.4f), %d visits" % (variant, K, sum(ms) / len(ms), min(ms), visits))
