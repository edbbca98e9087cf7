#!/usr/bin/env python
"""Developer tool: end-to-end frames/s of 8-bit RGB frames (tcrt_render_rgb8 & co.) against float32 frames, one process.

usage: python tools/e2e_rgb8.py [--rounds R] [--json PATH] [workload ...]

For every workload (default: the five BASELINE configs and two_mirrors_1080p_d50), float32 and RGB8 legs alternate
round after round on the same context and the same scene, each leg timed with the host clock around whole frames:
  blocking   tcrt_upload_scene + the blocking call into pinned host memory, one frame at a time (bench.py's e2e)
  async      tcrt_upload_scene + the async call into one of two pinned buffers, two frames in flight (bench.py's e2e_async)
  pageable   the blocking call into a plain numpy array (staged copy-out)
render_ms (tcrt_stats, CUDA events around the frame's launches) and d2h_ms (copy time not hidden behind them) are the
medians of the blocking leg's frames; RGB8 minus float render_ms is the cost of the quantisation launches.  With more
than one visible GPU the blocking and async legs also run through one in-process multi-device context.  Each workload
also gets a correctness line: the RGB8 frame equals quant8 of the float frame at full size.  Median and spread
(min..max) are over the rounds.
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

from bench import BASELINE_CONFIGS, WORKLOADS  # noqa: E402
from tilecoderaytracer_b200 import api  # noqa: E402

FORMATS = ("float32", "rgb8")


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out = [f"nvidia-smi unavailable: {e}"]
    return out


def quant8(c):
    return np.floor(np.clip(c.astype(np.float64), 0.0, 1.0) * 255.0 + 0.5).astype(np.uint8)


class Leg:
    """One context, one workload: the calls of a format."""

    def __init__(self, ctx, flat, camx, p, pinned_bytes):
        self.ctx, self.flat, self.camx, self.p = ctx, flat, camx, p
        w, h = p.width, p.height
        self.hb = [api.HostBuffer(pinned_bytes) for _ in range(2)]
        self.pinned = {"float32": [b.array(np.float32, (w, h, 3)) for b in self.hb],
                       "rgb8": [b.array(np.uint8, (w, h, 3)) for b in self.hb]}
        self.pageable = {"float32": np.empty((w, h, 3), np.float32), "rgb8": np.empty((w, h, 3), np.uint8)}

    def render(self, fmt, out):
        return self.ctx.render(self.p, out=out) if fmt == "float32" else self.ctx.render_rgb8(self.p, out=out)

    def submit(self, fmt, out):
        w = self.p.width
        return self.ctx.render_async(self.p, 0, w, out) if fmt == "float32" else self.ctx.render_async_rgb8(self.p, 0, w, out)

    def blocking(self, fmt, n):
        out = self.pinned[fmt][0]
        rms, d2h = [], []
        t0 = time.perf_counter()
        for _ in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            _, st = self.render(fmt, out)
            rms.append(max(st.render_ms))
            d2h.append(max(st.d2h_ms))
        return n / (time.perf_counter() - t0), statistics.median(rms), statistics.median(d2h)

    def in_flight(self, fmt, n):
        outs = self.pinned[fmt]
        t0 = time.perf_counter()
        tickets = []
        for i in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            tickets.append(self.submit(fmt, outs[i % 2]))
            if len(tickets) == 2:
                self.ctx.wait(tickets.pop(0))
        for t in tickets:
            self.ctx.wait(t)
        return n / (time.perf_counter() - t0)

    def paged(self, fmt, n):
        out = self.pageable[fmt]
        t0 = time.perf_counter()
        for _ in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            self.render(fmt, out)
        return n / (time.perf_counter() - t0)


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def fmt_cell(s, digits=1):
    return f"{s['median']:.{digits}f} ({s['min']:.{digits}f}..{s['max']:.{digits}f})"


def measure(name, rounds, n_gpus):
    scene_name, w, h, d = WORKLOADS[name]
    cam = api.Camera()
    # the library's scene builders print to the C stdout (e.g. SCENE 2's object count): to stderr, out of the report
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        scene = api.Scene().build(scene_name, cam)
    finally:
        ctypes.CDLL(None).fflush(None)               # what the C stdio buffered goes to stderr too
        os.dup2(saved, 1)
        os.close(saved)
    flat, camx = scene.flatten(), cam.export()
    p = api.default_params(w, h, d)
    ctx = api.Context([0])
    ctx.upload_flat(flat, camx)
    res = {"workload": name, "W": w, "H": h, "depth": d, "float_bytes": w * h * 12, "rgb8_bytes": w * h * 3}

    # ---- correctness at full size: RGB8 == quant8(float frame) ------------------------------------------------------
    img, st_f = ctx.render(p)
    got, st_8 = ctx.render_rgb8(p)
    bad = 0
    for c0 in range(0, w, 512):
        bad += int((got[c0:c0 + 512] != quant8(img[c0:c0 + 512])).any(-1).sum())
    res["correct"] = {"rgb8_equals_quant8_of_float": bad == 0, "pixels_differing": bad, "rays_equal": st_8.rays == st_f.rays,
                      "gpu_launches_float": st_f.gpu_launches, "gpu_launches_rgb8": st_8.gpu_launches}
    del img, got

    legs = [("1gpu", Leg(ctx, flat, camx, p, w * h * 12))]
    if n_gpus > 1:
        multi = api.Context(list(range(n_gpus)))
        multi.upload_flat(flat, camx)
        for _ in range(12):                        # the multi-device ctx re-cuts after every whole-frame render
            multi.render_device(p)
        legs.append((f"{n_gpus}gpu", Leg(multi, flat, camx, p, w * h * 12)))

    for tag, leg in legs:
        # warm-up of every call; the frame count of a timed window from the blocking float frame: >= ~0.5 s a window
        for fmt in FORMATS:
            leg.blocking(fmt, 2)
            leg.in_flight(fmt, 4)
        t0 = time.perf_counter()
        leg.blocking("float32", 3)
        frame_s = (time.perf_counter() - t0) / 3
        n = int(min(60, max(6, 0.5 / frame_s)))
        n_paged = int(min(20, max(3, 0.5 / frame_s / 2)))
        data = {f: {"blocking": [], "async": [], "pageable": [], "render_ms": [], "d2h_ms": []} for f in FORMATS}
        for r in range(rounds):
            order = FORMATS if r % 2 == 0 else FORMATS[::-1]
            for fmt in order:
                fps, rms, d2h = leg.blocking(fmt, n)
                data[fmt]["blocking"].append(fps)
                data[fmt]["render_ms"].append(rms)
                data[fmt]["d2h_ms"].append(d2h)
                data[fmt]["async"].append(leg.in_flight(fmt, n))
                if tag == "1gpu":
                    data[fmt]["pageable"].append(leg.paged(fmt, n_paged))
        out = {"frames_per_window": n, "frames_per_pageable_window": n_paged}
        for fmt in FORMATS:
            out[fmt] = {k: summary(v) for k, v in data[fmt].items() if v}
        out["quantise_ms"] = summary([a - b for a, b in zip(data["rgb8"]["render_ms"], data["float32"]["render_ms"])])
        res[tag] = out
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("workloads", nargs="*", default=BASELINE_CONFIGS + ["two_mirrors_1080p_d50"])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--json", default=None, help="write the results here as well")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    n_gpus = api.device_count()
    if n_gpus < 1:
        sys.exit("no CUDA device: this tool measures on the GPU and has no CPU path")
    info = {"devices": device_info(), "visible_gpus": n_gpus, "rounds": args.rounds, "results": []}
    print("device (name, power limit, max SM clock):", *info["devices"], sep="\n  ")
    print(f"visible GPUs: {n_gpus}; {args.rounds} rounds, float32 and RGB8 alternating; frames/s as median (min..max)")
    for name in args.workloads:
        r = measure(name, args.rounds, n_gpus)
        info["results"].append(r)
        c = r["correct"]
        print(f"\n== {name} ({r['W']}x{r['H']} d{r['depth']}; {r['float_bytes'] / 1e6:.1f} MB float32, "
              f"{r['rgb8_bytes'] / 1e6:.1f} MB RGB8 per frame)")
        print(f"  correct: RGB8 == quant8(float frame) at full size: {c['rgb8_equals_quant8_of_float']} "
              f"({c['pixels_differing']} pixels differ), rays equal: {c['rays_equal']}, "
              f"launches float {c['gpu_launches_float']} / RGB8 {c['gpu_launches_rgb8']}")
        for tag in [k for k in r if k.endswith("gpu")]:
            t = r[tag]
            for fmt in FORMATS:
                s = t[fmt]
                line = (f"  {tag:5s} {fmt:8s} blocking {fmt_cell(s['blocking'])}  async {fmt_cell(s['async'])}")
                if "pageable" in s:
                    line += f"  pageable {fmt_cell(s['pageable'])}"
                line += f"  render_ms {fmt_cell(s['render_ms'], 3)}  d2h_ms {fmt_cell(s['d2h_ms'], 3)}"
                print(line)
            print(f"  {tag:5s} quantise cost (RGB8 - float render_ms): {fmt_cell(t['quantise_ms'], 3)} ms")
        sys.stdout.flush()
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(info, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
