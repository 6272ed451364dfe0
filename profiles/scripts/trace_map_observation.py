"""B2S_TRACE timeline of one ICP.map_observation call on the course map (9999 scans x 360 beams) at 4 forced chunks,
after an untraced call of the same size."""
import math, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import b2slam
from b2slam import synth, _lib


def pinned(a):
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


room = synth.room_map_observation(9001, 9999, 360)
kr, hr = pinned(room["ranges"])
kp, hp = pinned(room["prior"])
icp = b2slam.ICP()
icp.set_static_map(room["obstacles_course"])
_lib.check(_lib.lib().b2s_tune(b"h2d_chunks", 4))
icp.map_observation(hr, hp, -math.pi, math.pi, clamp_inf_to=30.0, return_virtual=True)
print("== ICP.map_observation, 9999 scans x 360 beams, h2d_chunks 4", file=sys.stderr, flush=True)
os.environ["B2S_TRACE"] = "1"
icp.map_observation(hr, hp, -math.pi, math.pi, clamp_inf_to=30.0, return_virtual=True)
del os.environ["B2S_TRACE"]
_lib.check(_lib.lib().b2s_tune(b"h2d_chunks", 0))
