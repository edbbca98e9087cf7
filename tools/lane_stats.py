#!/usr/bin/env python
"""Developer tool: lane occupancy of the render kernel's phases (needs a -DTCRT_LANE_STATS build,
TCRT_LIB=<that library>).  usage: TCRT_LIB=.../libtcrt_stats.so python tools/lane_stats.py <workload>..."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import WORKLOADS  # noqa: E402
from tilecoderaytracer_b200 import _ffi, api  # noqa: E402

lib = _ffi.load()
NAMES = {0: "bounce iterations", 2: "nearest: inner-node steps", 4: "nearest: leaf phases", 6: "shadow: inner-node steps",
         8: "shadow: leaf phases", 10: "shadow sweeps (per light)", 12: "light loops"}
if "--wave" in sys.argv:
    NAMES = {2: "trace: inner-node steps", 4: "trace: leaf phases", 6: "trace: fetch events (lanes taking a task)",
             8: "trace: inner steps, lanes blocked on leaves", 12: "trace: inner steps, lanes without task"}
if "--pool" in sys.argv:
    NAMES = {0: "iterations", 2: "pool: inner-node steps", 4: "pool: leaf phases", 6: "pool: fetch events (free lanes)",
             8: "pool: inner steps, lanes blocked on leaves", 12: "pool: inner steps, lanes without task",
             10: "pool calls (light-A tasks)"}
if "--grid" in sys.argv:
    NAMES = {0: "nearest walks: DDA steps", 2: "shadow walks: DDA steps"}
ctx = api.Context([0])
for name in [a for a in sys.argv[1:] if not a.startswith("--")] or ["synth256_1080p_d10"]:
    scene_name, w, h, d = WORKLOADS[name]
    cam = api.Camera()
    scene = api.Scene().build(scene_name, cam)
    ctx.upload(scene, cam)
    p = api.default_params(w, h, d)
    ctx.render_device(p)
    out = (C.c_ulonglong * 16)()
    fn = lib.tcrt_dev_lane_stats_grid if "--grid" in sys.argv else lib.tcrt_dev_lane_stats_pool if "--pool" in sys.argv else (lib.tcrt_dev_lane_stats_wave if "--wave" in sys.argv else lib.tcrt_dev_lane_stats)
    fn(out, 1)
    st = ctx.render_device(p)
    fn(out, 0)
    print(f"== {name}: {st.render_ms[0]:.3f} ms, {st.rays} rays")
    for k, label in NAMES.items():
        n, lanes = out[k], out[k + 1]
        if n:
            print(f"  {label:28s} warp-steps {n:12d}  lanes/step {lanes / n:5.2f}")
    if "--grid" in sys.argv:
        print(f"  shadow walks of a bounce: sum over passes of the longest walk {out[4]}, longest per-lane sum {out[5]} "
              f"({out[5] / max(out[4], 1):.3f})")
        print(f"  light passes at dead levels (DESIGN.md §4.1c): warp-passes skipped whole {out[6]}, lane-passes {out[7]} "
              f"({out[7] / max(st.rays_shadow, 1):.3f} of the {st.rays_shadow} shadow rays counted)")
