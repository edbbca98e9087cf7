#!/usr/bin/env python
"""Developer tool: cost of the primary-hit buffers (tcrt_hit_buffers) and of picking (tcrt_pick), one process, one GPU.

usage: python tools/e2e_hits.py [--reps N] [--json PATH] [workload ...]

For every workload (default: default_1080p_d5, default_4k_d50, synth256_8k_d10, synth1024_4k_d50, two_mirrors_1080p_d50):
  kernel      render_ms of the device-only call (CUDA events around the hit kernel) against render_ms of the device-only
              float frame (tcrt_render_device: one render launch) of the same workload
  e2e         host clock around whole blocking tcrt_hit_buffers calls into pinned and into pageable memory, with all three
              buffers (20 B/pixel) and with `object` only (4 B/pixel); GB/s = bytes copied back / e2e time
  pick        host clock around tcrt_pick of 1, 1024 and 1 M random pixels
Every number is the median (min..max) over --reps calls after one warm-up call.  A correctness line checks that picks at
random pixels equal the buffers there.  Multi-device contexts are not measured here.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402

from bench import WORKLOADS  # noqa: E402
from tilecoderaytracer_b200 import api  # noqa: E402

DEFAULT = ["default_1080p_d5", "default_4k_d50", "synth256_8k_d10", "synth1024_4k_d50", "two_mirrors_1080p_d50"]
NAMES = ("object", "distance", "normal")
BPP = {"object": 4, "distance": 4, "normal": 12}


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out = [f"nvidia-smi unavailable: {e}"]
    return out


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def cell(s, digits=2):
    return f"{s['median']:.{digits}f} ({s['min']:.{digits}f}..{s['max']:.{digits}f})"


def timed(fn, reps):
    fn()                                            # warm-up: module load, buffer allocation
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return summary(ms)


def build_scene(name):
    scene_name, w, h, d = WORKLOADS[name]
    cam = api.Camera()
    # the library's scene builders print to the C stdout (e.g. SCENE 2's object count): to stderr, out of the report
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        scene = api.Scene().build(scene_name, cam)
    finally:
        ctypes.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)
    return scene, scene.flatten(), cam.export(), api.default_params(w, h, d)   # the flat arrays live in `scene`


def measure(name, reps):
    scene, flat, camx, p = build_scene(name)
    w, h = p.width, p.height
    n = w * h
    ctx = api.Context([0])
    ctx.upload_flat(flat, camx)
    res = {"workload": name, "W": w, "H": h, "depth": p.max_depth, "bytes_all": n * 20, "bytes_object": n * 4}

    # ---- kernels: hit kernel against the float frame's render launch --------------------------------------------------
    frame_ms, hit_ms = [], []
    ctx.render_device(p)
    ctx.hit_buffers_device(p)
    for _ in range(reps):
        frame_ms.append(ctx.render_device(p).render_ms[0])
        hit_ms.append(ctx.hit_buffers_device(p).render_ms[0])
    res["frame_render_ms"] = summary(frame_ms)
    res["hit_kernel_ms"] = summary(hit_ms)

    # ---- end to end into host memory ---------------------------------------------------------------------------------
    hb = {k: api.HostBuffer(n * BPP[k]) for k in NAMES}
    pinned = {"object": hb["object"].array(np.int32, (w, h)), "distance": hb["distance"].array(np.float32, (w, h)),
              "normal": hb["normal"].array(np.float32, (w, h, 3))}
    pageable = {"object": np.empty((w, h), np.int32), "distance": np.empty((w, h), np.float32),
                "normal": np.empty((w, h, 3), np.float32)}
    res["e2e"] = {}
    for kind, bufs in (("pinned", pinned), ("pageable", pageable)):
        for sel in ("all", "object"):
            out = bufs if sel == "all" else {"object": bufs["object"]}
            d2h = []

            def call(out=out, d2h=d2h):
                _, st = ctx.hit_buffers(p, out=out)
                d2h.append(st.d2h_ms[0])

            s = timed(call, reps)
            nbytes = res["bytes_all"] if sel == "all" else res["bytes_object"]
            s["GB_per_s"] = nbytes / (s["median"] * 1e-3) / 1e9
            s["d2h_ms_median"] = statistics.median(d2h[1:])
            res["e2e"][f"{kind}_{sel}"] = s

    # ---- correctness: picks equal the buffers -------------------------------------------------------------------------
    got, _ = ctx.hit_buffers(p)
    rng = np.random.default_rng(1)
    xs, zs = rng.integers(0, w, 4096), rng.integers(0, h, 4096)
    o, d, nn = ctx.pick(p, xs, zs)
    res["correct"] = {"pick_equals_buffers": bool(np.array_equal(o, got["object"][xs, zs])
                                                  and np.array_equal(d.view(np.uint32), got["distance"][xs, zs].view(np.uint32))
                                                  and np.array_equal(nn.view(np.uint32), got["normal"][xs, zs].view(np.uint32))),
                      "miss_fraction": float((got["object"] < 0).mean())}
    del got

    # ---- picking latency ------------------------------------------------------------------------------------------------
    res["pick_ms"] = {}
    for k in (1, 1024, 1 << 20):
        px, pz = rng.integers(0, w, k), rng.integers(0, h, k)
        res["pick_ms"][str(k)] = timed(lambda px=px, pz=pz: ctx.pick(p, px, pz), reps)
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    info = device_info()
    print("# device:", "; ".join(info))
    results = []
    for name in a.workloads:
        r = measure(name, a.reps)
        results.append(r)
        print(f"\n## {name} ({r['W']}x{r['H']} d{r['depth']}): {r['bytes_all'] / 1e6:.1f} MB all buffers, "
              f"{r['bytes_object'] / 1e6:.1f} MB object only; correct: {r['correct']}")
        print(f"kernel ms: hit {cell(r['hit_kernel_ms'], 3)}   float frame render {cell(r['frame_render_ms'], 3)}")
        for key, s in r["e2e"].items():
            print(f"e2e {key:16s} ms {cell(s, 3)}  {s['GB_per_s']:.1f} GB/s  (d2h_ms {s['d2h_ms_median']:.3f})")
        for k, s in r["pick_ms"].items():
            print(f"pick {k:>8s} px  ms {cell(s, 3)}")
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"device": info, "reps": a.reps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
