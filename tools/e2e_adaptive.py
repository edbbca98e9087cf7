#!/usr/bin/env python
"""Developer tool: adaptive anti-aliased frames (tcrt_render_columns_adaptive & co.) end to end, one process.

usage: python tools/e2e_adaptive.py [--rounds R] [--json PATH] [--ss 2,4] [--contrast 0,8,32] [--no-profile] [workload ...]

For every workload (default: default_1080p_d5, default_4k_d50, two_mirrors_1080p_d50, synth256_4k_d10, synth256_8k_d10)
and every ss, these legs alternate round after round on one context and one scene, each a window of blocking frames into
pinned host memory timed with the host clock:
  plain          tcrt_render_columns (the frame without anti-aliasing)
  ss             tcrt_render_columns_ss (every pixel supersampled)
  adaptive f32   tcrt_render_columns_adaptive at each contrast
  adaptive rgb8  tcrt_render_columns_adaptive_rgb8 at each contrast
frames/s are medians (min..max) over the rounds; render_ms (tcrt_stats: CUDA events from a frame's first launch to its
last, for an adaptive frame including the wait for the list's length) is the median over the frames.  Per (workload, ss,
contrast): the refined fraction, the primary rays against the plain frame's, the speed-up of the adaptive frame over
render_ss (blocking float frames), and a correctness line (the adaptive frame equals where(mask, render_ss, render) bit for
bit, n_refined equals the mask's sum).  Unless --no-profile, one adaptive float frame per combination is traced with
torch.profiler (a separate pass, after the timed ones) and its kernel time is split by kernel: plain pass (render_kernel /
render_grid_kernel), classify (classify + scan + compact), sample pass (the list-mode render kernels), resolve, and other
kernels (the driver's memsets).  Kernels of different render streams overlap, so the split is a sum of kernel times, not of
wall time.
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

from tilecoderaytracer_b200 import api  # noqa: E402

WORKLOADS = {
    "default_1080p_d5": ("default", 1920, 1080, 5),
    "default_4k_d50": ("default", 3840, 2160, 50),
    "two_mirrors_1080p_d50": ("two_mirrors", 1920, 1080, 50),
    "synth256_4k_d10": ("synth256", 3840, 2160, 10),
    "synth256_8k_d10": ("synth256", 7680, 4320, 10),
}


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out = [f"nvidia-smi unavailable: {e}"]
    return out


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def cell(s, digits=1):
    return f"{s['median']:.{digits}f} ({s['min']:.{digits}f}..{s['max']:.{digits}f})"


def quiet_scene(name, cam):
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        return api.Scene().build(name, cam)
    finally:
        ctypes.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)


def quant8(c):
    return np.floor(np.clip(np.nan_to_num(c.astype(np.float64), nan=0.0), 0.0, 1.0) * 255.0 + 0.5).astype(np.int16)


def refine_mask(frame, contrast):
    """The contract of include/tcrt.h (the same restatement as tests/test_adaptive_frames.py)."""
    q = quant8(frame)
    W, H, _ = q.shape
    if contrast < 0:
        return np.ones((W, H), bool)
    m = np.zeros((W, H), bool)
    for dx in (-1, 0, 1):
        for dz in (-1, 0, 1):
            if dx or dz:
                xs, xd = slice(max(0, -dx), W - max(0, dx)), slice(max(0, dx), W - max(0, -dx))
                zs, zd = slice(max(0, -dz), H - max(0, dz)), slice(max(0, dz), H - max(0, -dz))
                m[xs, zs] |= np.abs(q[xs, zs] - q[xd, zd]).max(-1) > contrast
    return m


class Legs:
    def __init__(self, ctx, flat, camx, p, ss):
        self.ctx, self.flat, self.camx, self.p, self.ss = ctx, flat, camx, p, ss
        w, h = p.width, p.height
        self.hb = api.HostBuffer(w * h * 12)
        self.f32 = self.hb.array(np.float32, (w, h, 3))
        self.u8 = self.hb.array(np.uint8, (w, h, 3))

    def frame(self, leg, contrast=None):
        if leg == "plain":
            return self.ctx.render(self.p, out=self.f32)[1]
        if leg == "ss":
            return self.ctx.render_ss(self.p, self.ss, out=self.f32)[1]
        if leg == "adaptive_f32":
            return self.ctx.render_adaptive(self.p, self.ss, contrast, out=self.f32)[3]
        return self.ctx.render_adaptive_rgb8(self.p, self.ss, contrast, out=self.u8)[3]

    def window(self, leg, n, contrast=None):
        rms = []
        t0 = time.perf_counter()
        for _ in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            rms.append(max(self.frame(leg, contrast).render_ms))
        return n / (time.perf_counter() - t0), statistics.median(rms)


def phase_split(ctx, p, ss, contrast):
    """Kernel time of one adaptive float frame by phase, from a torch.profiler trace (CUPTI sees the library's kernels)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    ctx.render_adaptive_device(p, ss, contrast)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.render_adaptive_device(p, ss, contrast)
        torch.cuda.synchronize()
    phases = {"plain": 0.0, "classify": 0.0, "sample": 0.0, "resolve": 0.0, "other": 0.0}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name, us = ev.name, ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "resolve_list" in name:
            k = "resolve"
        elif "list_kernel" in name:
            k = "sample"
        elif "render_kernel" in name or "render_grid_kernel" in name:
            k = "plain"
        elif any(s in name for s in ("classify_kernel", "scan_kernel", "compact_kernel")):
            k = "classify"
        else:
            k = "other"
        phases[k] += us / 1000.0
    return phases


def measure(name, ss, contrasts, rounds, profile_on):
    scene_name, w, h, d = WORKLOADS[name]
    cam = api.Camera()
    scene = quiet_scene(scene_name, cam)
    flat, camx = scene.flatten(), cam.export()
    p = api.default_params(w, h, d)
    ctx = api.Context([0])
    ctx.upload_flat(flat, camx)
    legs = Legs(ctx, flat, camx, p, ss)
    res = {"workload": name, "W": w, "H": h, "depth": d, "ss": ss, "contrast": {}}
    # correctness and counts, from the frames themselves
    plain, st_plain = ctx.render(p)
    plain = plain.copy()
    full, st_ss = ctx.render_ss(p, ss)
    full = full.copy()
    res["plain_rays_primary"], res["ss_rays_primary"] = st_plain.rays_primary, st_ss.rays_primary
    for c in contrasts:
        mask = refine_mask(plain, c)
        got, gmask, n, st = ctx.render_adaptive(p, ss, c, mask=np.empty((w, h), np.uint8))
        want = np.where(mask[..., None], full, plain)
        bad = int((got.view(np.uint32) != want.view(np.uint32)).any(-1).sum())
        res["contrast"][c] = {"n_refined": n, "fraction": n / (w * h), "mask_sum": int(mask.sum()),
                              "mask_equal": bool(np.array_equal(gmask, mask.astype(np.uint8))), "pixels_differing": bad,
                              "rays_primary": st.rays_primary, "rays": st.rays, "gpu_launches": st.gpu_launches}
    del plain, full, got, want
    # warm-up of every leg, then windows sized to ~0.3 s of the slowest leg (render_ss)
    for leg in ("plain", "ss"):
        legs.window(leg, 1)
    for c in contrasts:
        legs.window("adaptive_f32", 1, c)
        legs.window("adaptive_rgb8", 1, c)
    t0 = time.perf_counter()
    legs.window("ss", 1)
    n = int(min(20, max(3, 0.3 / (time.perf_counter() - t0))))
    keys = [("plain", None), ("ss", None)] + [(k, c) for c in contrasts for k in ("adaptive_f32", "adaptive_rgb8")]
    data = {k: {"fps": [], "render_ms": []} for k in keys}
    for r in range(rounds):
        for k in (keys if r % 2 == 0 else keys[::-1]):
            fps, rms = legs.window(k[0], n, k[1])
            data[k]["fps"].append(fps)
            data[k]["render_ms"].append(rms)
    res["frames_per_window"] = n
    res["plain"] = {m: summary(v) for m, v in data[("plain", None)].items()}
    res["ss_full"] = {m: summary(v) for m, v in data[("ss", None)].items()}
    for c in contrasts:
        rc = res["contrast"][c]
        for k in ("adaptive_f32", "adaptive_rgb8"):
            rc[k] = {m: summary(v) for m, v in data[(k, c)].items()}
        rc["speedup_over_ss"] = rc["adaptive_f32"]["fps"]["median"] / res["ss_full"]["fps"]["median"]
        if profile_on:
            try:
                rc["kernel_ms"] = phase_split(ctx, p, ss, c)
            except Exception as e:          # the timed legs stand without the split
                rc["kernel_ms"] = {"error": repr(e)}
    del legs
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("workloads", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--ss", default="2,4")
    ap.add_argument("--contrast", default="0,8,32")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    n_gpus = api.device_count()
    if n_gpus < 1:
        sys.exit("no CUDA device: this tool measures on the GPU and has no CPU path")
    contrasts = [int(c) for c in args.contrast.split(",")]
    info = {"devices": device_info(), "visible_gpus": n_gpus, "rounds": args.rounds, "results": []}
    print("device (name, power limit, max SM clock, current SM clock):", *info["devices"], sep="\n  ")
    print(f"{args.rounds} rounds, legs alternating, blocking frames into pinned host memory; frames/s as median (min..max)")
    for name in args.workloads:
        for ss in (int(s) for s in args.ss.split(",")):
            r = measure(name, ss, contrasts, args.rounds, not args.no_profile)
            info["results"].append(r)
            print(f"\n== {name} ({r['W']}x{r['H']} d{r['depth']}) ss={ss}")
            print(f"  plain    {cell(r['plain']['fps'])} f/s  render_ms {cell(r['plain']['render_ms'], 3)}  "
                  f"primary rays {r['plain_rays_primary']}")
            print(f"  ss       {cell(r['ss_full']['fps'])} f/s  render_ms {cell(r['ss_full']['render_ms'], 3)}  "
                  f"primary rays {r['ss_rays_primary']}")
            for c in contrasts:
                rc = r["contrast"][c]
                ok = rc["pixels_differing"] == 0 and rc["mask_equal"] and rc["n_refined"] == rc["mask_sum"]
                print(f"  contrast {c:3d}: refined {100 * rc['fraction']:.2f} % ({rc['n_refined']}), primary rays "
                      f"{rc['rays_primary'] / r['plain_rays_primary']:.2f} plain frames, {rc['gpu_launches']} launches; "
                      f"{'bit-identical' if ok else 'MISMATCH: ' + str(rc['pixels_differing']) + ' pixels'}")
                for k in ("adaptive_f32", "adaptive_rgb8"):
                    print(f"    {k:13s} {cell(rc[k]['fps'])} f/s  render_ms {cell(rc[k]['render_ms'], 3)}")
                print(f"    speed-up over render_ss (float): {rc['speedup_over_ss']:.2f}x")
                km = rc.get("kernel_ms")
                if km and "error" not in km:
                    print("    kernel ms: " + "  ".join(f"{k} {v:.3f}" for k, v in km.items()))
                elif km:
                    print(f"    kernel ms: not measured ({km['error']})")
            sys.stdout.flush()
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(info, f, indent=1, default=str)
            f.write("\n")


if __name__ == "__main__":
    main()
