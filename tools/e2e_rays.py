#!/usr/bin/env python
"""Developer tool: cost of ray batches (tcrt_trace_rays and its device form), one process, one GPU.

usage: python tools/e2e_rays.py [--reps N] [--json PATH] [workload ...]

For every workload (default: default_4k_d50, synth256_8k_d10, two_mirrors_1080p_d50, synth1024_4k_d50) the batch is the
frame's eye rays, built in numpy float32 as tests/test_ray_batches.py builds them, so every batch equals the frame:
  kernel   render_ms of tcrt_trace_rays_device (CUDA events around the batch's launches; inputs and outputs in device
           memory) against render_ms of tcrt_render_device (the band kernel) for the same frame, the L2 overwritten before
           every call.  Eye rays in three orders: "tile" (the band kernel's 4x8-tile claim order), "x" (x-major, the frame's
           layout) and "shuffle" (a fixed random permutation: no coherence left in a warp).
  e2e      host clock around whole blocking calls, tile order: host forms with pinned and pageable inputs and outputs,
           per-ray and shared origins, and the device form; bus GB/s = bytes in + bytes out / e2e time.
Every number is the median (min..max) over --reps calls after one warm-up call.  A correctness line checks that each
ordering reproduces the frame bit for bit.  Multi-device contexts are not measured here.
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

DEFAULT = ["default_4k_d50", "synth256_8k_d10", "two_mirrors_1080p_d50", "synth1024_4k_d50"]
F32 = np.float32


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
    sys.stdout.flush()                              # the scene builders print to the C stdout: to stderr, out of the report
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        scene = api.Scene().build(scene_name, cam)
    finally:
        ctypes.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)
    return scene, scene.flatten(), cam.export(), api.default_params(w, h, d)


def eye_rays(cam, w, h, order):
    """Directions of the frame's primary rays in `order` and the pixel index x*H + z of each."""
    x, z = np.meshgrid(np.arange(w), np.arange(h), indexing="ij")
    x, z = x.ravel(), z.ravel()
    if order == "tile":
        t, i = np.divmod(np.arange(w * h), 32)
        tx, tz = np.divmod(t, h // 8)
        x, z = tx * 4 + i % 4, tz * 8 + i // 4
    elif order == "shuffle":
        perm = np.random.default_rng(7).permutation(w * h)
        x, z = x[perm], z[perm]
    sx = (x.astype(F32) / F32(w)) * F32(cam.screen_width) - F32(cam.screen_halfwidth)
    sy = (z.astype(F32) / F32(h)) * F32(cam.screen_height) - F32(cam.screen_halfheight)
    so, hz, vt = (np.array(v[:], F32) for v in (cam.screen_origin, cam.horizontal, cam.vertical))
    pixel = (so + hz * sx[:, None]) + vt * sy[:, None]
    return np.ascontiguousarray(api.normalize_like_reference(pixel - np.array(cam.eye[:], F32))), x * h + z


def measure(name, reps):
    import torch

    scene, flat, camx, p = build_scene(name)
    w, h = p.width, p.height
    n = w * h
    ctx = api.Context([0])
    ctx.upload_flat(flat, camx)
    dev = torch.device("cuda:0")
    eye = np.array(camx.eye[:], F32)
    res = {"workload": name, "W": w, "H": h, "depth": p.max_depth, "rays": n}

    # ---- kernels: ray mode against band mode ---------------------------------------------------------------------------
    frame = torch.empty((n, 3), dtype=torch.float32, device=dev)
    ctx.render_device(p)
    band = []
    for _ in range(reps):
        ctx.flush_l2()
        band.append(ctx.render_device(p).render_ms[0])
    res["band_kernel_ms"] = summary(band)
    ref = np.empty((w, h, 3), F32)
    ctx.download(ref)
    ref = ref.reshape(n, 3)
    res["ray_kernel_ms"], res["correct"] = {}, {}
    t_eye = torch.from_numpy(eye).to(dev)
    for order in ("tile", "x", "shuffle"):
        d, pix = eye_rays(camx, w, h, order)
        t_d = torch.from_numpy(d).to(dev)
        del d
        torch.cuda.synchronize()
        ms = []
        ctx.trace_rays_device(p, n, t_eye.data_ptr(), t_d.data_ptr(), frame.data_ptr(), shared_origin=True)
        for _ in range(reps):
            ctx.flush_l2()
            _, st = ctx.trace_rays_device(p, n, t_eye.data_ptr(), t_d.data_ptr(), frame.data_ptr(), shared_origin=True)
            ms.append(st.render_ms[0])
        res["ray_kernel_ms"][order] = summary(ms)
        got = frame.cpu().numpy()
        res["correct"][order] = bool(np.array_equal(got.view(np.uint32), ref[pix].view(np.uint32)))
        del t_d, got

    # ---- end to end, tile order ------------------------------------------------------------------------------------------
    d, _ = eye_rays(camx, w, h, "tile")
    o = np.ascontiguousarray(np.broadcast_to(eye, d.shape))
    hb = [api.HostBuffer(n * 12) for _ in range(3)]
    pinned_o, pinned_d, pinned_rgb = (b.array(F32, (n, 3)) for b in hb)
    pinned_o[:], pinned_d[:] = o, d
    pageable_rgb = np.empty((n, 3), F32)
    res["e2e"] = {}
    cases = [("pinned per-ray origins", pinned_o, pinned_d, pinned_rgb, 24),
             ("pinned shared origin", eye, pinned_d, pinned_rgb, 12),
             ("pageable per-ray origins", o, d, pageable_rgb, 24),
             ("pageable shared origin", eye, d, pageable_rgb, 12)]
    for key, oo, dd, out, in_b in cases:
        d2h = []

        def call(oo=oo, dd=dd, out=out, d2h=d2h):
            _, _, st = ctx.trace_rays(p, oo, dd, out=out)
            d2h.append(st.d2h_ms[0])

        s = timed(call, reps)
        s["bytes"] = n * (in_b + 12)
        s["GB_per_s"] = s["bytes"] / (s["median"] * 1e-3) / 1e9
        s["d2h_ms_median"] = statistics.median(d2h[1:])
        res["e2e"][key] = s
    t_o, t_d = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    torch.cuda.synchronize()
    s = timed(lambda: ctx.trace_rays_device(p, n, t_o.data_ptr(), t_d.data_ptr(), frame.data_ptr()), reps)
    s["bytes"], s["GB_per_s"] = 0, 0.0
    res["e2e"]["device form per-ray origins"] = s
    del t_o, t_d, frame
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    info = device_info()
    print("# device:", "; ".join(info))
    results = []
    for name in a.workloads:
        r = measure(name, a.reps)
        results.append(r)
        print(f"\n## {name} ({r['W']}x{r['H']} d{r['depth']}, {r['rays'] / 1e6:.2f} M rays); bit-identical to the frame: "
              f"{r['correct']}")
        band = r["band_kernel_ms"]["median"]
        print(f"kernel ms: band mode {cell(r['band_kernel_ms'], 3)}")
        for order, s in r["ray_kernel_ms"].items():
            print(f"kernel ms: ray mode, {order:8s} {cell(s, 3)}  {s['median'] / band:.3f}x band")
        for key, s in r["e2e"].items():
            print(f"e2e {key:30s} ms {cell(s, 2)}  {s['GB_per_s']:.1f} GB/s over the bus"
                  + (f"  (d2h_ms {s['d2h_ms_median']:.2f})" if "d2h_ms_median" in s else ""))
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"device": info, "reps": a.reps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
