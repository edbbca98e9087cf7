#!/usr/bin/env python
"""Developer tool: cost of the occlusion queries (tcrt_occluded_lights, tcrt_occluded_rays and their device forms), one
process, one GPU.

usage: python tools/e2e_occlusion.py [--reps N] [--json PATH] [workload ...]

For every workload (default: default_4k_d50, synth256_8k_d10, two_mirrors_1080p_d50, boxes_4k_d12):
  points   render_ms of tcrt_occluded_lights_device for one point per pixel — the primary hit points of the frame's non-light
           hits, t*D + O + 1e-3*normal from the hit buffers, in the band kernel's 4x8-tile order — against render_ms of
           tcrt_render_device (the band kernel) for the same frame.  Every point is tested against every light.
  rays     render_ms of tcrt_occluded_rays_device with tmax = +inf against tcrt_intersect_rays_device on the same eye rays
           (shared origin, tile order), with all three hit outputs and with the object only.
  e2e      host clock around whole blocking calls of both host forms: pinned and pageable inputs and outputs.
Kernel times have the L2 overwritten before every call.  Every number is the median (min..max) over --reps calls after one
warm-up call.  Multi-device contexts are not measured here.
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

OWN = {"boxes_4k_d12": ("boxes:3:14", 3840, 2160, 12)}
DEFAULT = ["default_4k_d50", "synth256_8k_d10", "two_mirrors_1080p_d50", "boxes_4k_d12"]
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


def kernel_ms(ctx, fn, reps):
    fn()
    ms = []
    for _ in range(reps):
        ctx.flush_l2()
        ms.append(fn().render_ms[0])
    return summary(ms)


def build_scene(name):
    scene_name, w, h, d = OWN.get(name) or WORKLOADS[name]
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


def tile_order(w, h):
    """Pixel index x*H + z of queue position q in the band kernel's 4x8-tile order."""
    t, i = np.divmod(np.arange(w * h), 32)
    tx, tz = np.divmod(t, h // 8)
    return (tx * 4 + i % 4) * h + tz * 8 + i // 4


def eye_dirs(cam, w, h, pix):
    x, z = np.divmod(pix, h)
    sx = (x.astype(F32) / F32(w)) * F32(cam.screen_width) - F32(cam.screen_halfwidth)
    sy = (z.astype(F32) / F32(h)) * F32(cam.screen_height) - F32(cam.screen_halfheight)
    so, hz, vt = (np.array(v[:], F32) for v in (cam.screen_origin, cam.horizontal, cam.vertical))
    pixel = (so + hz * sx[:, None]) + vt * sy[:, None]
    return np.ascontiguousarray(api.normalize_like_reference(pixel - np.array(cam.eye[:], F32)))


def measure(name, reps):
    import torch

    scene, flat, camx, p = build_scene(name)
    w, h = p.width, p.height
    n = w * h
    ctx = api.Context([0])
    ctx.upload_flat(flat, camx)
    dev = torch.device("cuda:0")
    eye = np.array(camx.eye[:], F32)
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    res = {"workload": name, "W": w, "H": h, "depth": p.max_depth, "pixels": n, "lights": flat.n_lights,
           "dispatch": ctx.scene_structures()}
    res["render_kernel_ms"] = kernel_ms(ctx, lambda: ctx.render_device(p), reps)

    # ---- the frame's primary hit points, tile order ---------------------------------------------------------------------
    pix = tile_order(w, h)
    d = eye_dirs(camx, w, h, pix)
    hb, _ = ctx.hit_buffers(api.default_params(w, h, 0))
    obj = hb["object"].reshape(-1)[pix]
    t = hb["distance"].reshape(-1)[pix]
    nrm = hb["normal"].reshape(-1, 3)[pix]
    keep = obj >= 0
    keep[keep] &= info[obj[keep], 2] == 0
    pts = np.ascontiguousarray(((d[keep] * t[keep, None]) + eye) + nrm[keep] * F32(1e-3), F32)
    del hb, obj, t, nrm
    m = len(pts)
    res["points"] = m
    t_p = torch.from_numpy(pts).to(dev)
    t_occ = torch.empty(max(1, m * flat.n_lights), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    res["points_kernel_ms"] = kernel_ms(ctx, lambda: ctx.occluded_lights_device(m, t_p.data_ptr(), t_occ.data_ptr())[1], reps)
    _, st = ctx.occluded_lights_device(m, t_p.data_ptr(), t_occ.data_ptr())
    occ = t_occ.cpu().numpy()[:m * flat.n_lights]
    res["points_tests"] = int(st.rays_shadow)
    res["points_occluded_share"] = float((occ == 1).mean()) if m else 0.0
    res["points_invalid"] = int((occ == 0xFF).sum())
    del t_p, t_occ

    # ---- eye rays, tmax = +inf, against their nearest hits ----------------------------------------------------------------
    t_e = torch.from_numpy(eye).to(dev)
    t_d = torch.from_numpy(d).to(dev)
    t_t = torch.full((n,), float("inf"), dtype=torch.float32, device=dev)
    t_o = torch.empty(n, dtype=torch.uint8, device=dev)
    t_obj = torch.empty(n, dtype=torch.int32, device=dev)
    t_dist = torch.empty(n, dtype=torch.float32, device=dev)
    t_n = torch.empty((n, 3), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    p0 = api.default_params(1, 1, 0)
    res["occluded_rays_kernel_ms"] = kernel_ms(
        ctx, lambda: ctx.occluded_rays_device(n, t_e.data_ptr(), t_d.data_ptr(), t_t.data_ptr(), t_o.data_ptr(),
                                              shared_origin=True)[1], reps)
    res["intersect_rays_kernel_ms"] = kernel_ms(
        ctx, lambda: ctx.intersect_rays_device(p0, n, t_e.data_ptr(), t_d.data_ptr(), t_obj.data_ptr(), t_dist.data_ptr(),
                                               t_n.data_ptr(), shared_origin=True)[1], reps)
    res["intersect_rays_object_only_kernel_ms"] = kernel_ms(
        ctx, lambda: ctx.intersect_rays_device(p0, n, t_e.data_ptr(), t_d.data_ptr(), t_obj.data_ptr(), shared_origin=True)[1],
        reps)
    res["rays_occluded_share"] = float((t_o.cpu().numpy() == 1).mean())
    del t_e, t_d, t_t, t_o, t_obj, t_dist, t_n
    torch.cuda.empty_cache()

    # ---- end to end: pinned against pageable ------------------------------------------------------------------------------
    nl = flat.n_lights
    hbuf = [api.HostBuffer(max(1, k)) for k in (m * 12, m * nl, n * 12, n * 4, n)]
    pin_p = hbuf[0].array(F32, (m, 3))
    pin_lo = hbuf[1].array(np.uint8, (m, nl))
    pin_d = hbuf[2].array(F32, (n, 3))
    pin_t = hbuf[3].array(F32, (n,))
    pin_ro = hbuf[4].array(np.uint8, (n,))
    pin_p[:], pin_d[:], pin_t[:] = pts, d, np.inf
    tinf = np.full(n, np.inf, F32)
    res["e2e"] = {}
    cases = [("lights pinned", lambda: ctx.occluded_lights(pin_p, out=pin_lo), m * (12 + nl)),
             ("lights pageable", lambda: ctx.occluded_lights(pts), m * (12 + nl)),
             ("rays pinned shared origin", lambda: ctx.occluded_rays(eye, pin_d, pin_t, out=pin_ro), n * 17),
             ("rays pageable shared origin", lambda: ctx.occluded_rays(eye, d, tinf), n * 17)]
    for key, fn, nbytes in cases:
        s = timed(fn, reps)
        s["bytes"] = nbytes
        s["GB_per_s"] = nbytes / (s["median"] * 1e-3) / 1e9
        res["e2e"][key] = s
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
        print(f"\n## {name} ({r['W']}x{r['H']} d{r['depth']}, {r['lights']} lights, {r['points']} hit points of "
              f"{r['pixels']} pixels)")
        rk = r["render_kernel_ms"]["median"]
        print(f"kernel ms: render launch of the frame   {cell(r['render_kernel_ms'], 3)}")
        print(f"kernel ms: occluded_lights, hit points  {cell(r['points_kernel_ms'], 3)}  {r['points_kernel_ms']['median'] / rk:.3f}x"
              f" render  ({r['points_tests']} tests, {100 * r['points_occluded_share']:.1f} % occluded,"
              f" {r['points_invalid']} invalid)")
        ik = r["intersect_rays_kernel_ms"]["median"]
        print(f"kernel ms: intersect_rays, eye rays     {cell(r['intersect_rays_kernel_ms'], 3)}")
        print(f"kernel ms: intersect_rays, object only  {cell(r['intersect_rays_object_only_kernel_ms'], 3)}")
        print(f"kernel ms: occluded_rays, tmax = +inf   {cell(r['occluded_rays_kernel_ms'], 3)}  "
              f"{r['occluded_rays_kernel_ms']['median'] / ik:.3f}x intersect  ({100 * r['rays_occluded_share']:.1f} % occluded)")
        for key, s in r["e2e"].items():
            print(f"e2e {key:30s} ms {cell(s, 2)}  {s['GB_per_s']:.1f} GB/s over the bus")
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"device": info, "reps": a.reps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
