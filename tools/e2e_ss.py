#!/usr/bin/env python
"""Developer tool: supersampled frames (tcrt_render_columns_ss & co.) end to end, one process.

usage: python tools/e2e_ss.py [--rounds R] [--json PATH] [--ss 1,2,4] [workload ...]

For every workload (default: default_1080p_d5, default_4k_d50, synth256_8k_d10) and every ss, these legs alternate round
after round on one context and one scene, each timed with the host clock around whole frames:
  ss float / ss rgb8     tcrt_upload_scene + the supersampled call into pinned host memory: blocking (one frame at a
                         time) and async (two frames in flight)
  sample                 the plain tcrt_render_columns of the sample frame (ss*W x ss*H) into pinned host memory, blocking
  workaround             the same sample frame plus the box average in numpy on the host: what a user without
                         supersampled frames does
frames/s are medians (min..max) over the rounds; Gsamples/s = frames/s * ss*ss*W*H / 1e9 (primary rays).  render_ms
(tcrt_stats, CUDA events around the frame's launches) is the median over the blocking frames; ss float minus sample
render_ms is the cost of the resolve launches and the scratch round trip.  A sample frame above --max-host-gb of host
memory is not copied out: its sample leg is the device-only call (one launch) and its workaround is not measured.
Each combination gets a correctness line: column ranges of the supersampled frame equal resolve() of the plain render of
the matching sample columns, bit for bit.  With more than one visible GPU the blocking ss float leg also runs through one
in-process multi-device context.
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

DEFAULT_WORKLOADS = ["default_1080p_d5", "default_4k_d50", "synth256_8k_d10"]


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out = [f"nvidia-smi unavailable: {e}"]
    return out


def resolve(samples, ss):
    """The order of tcrt.h: acc = sample(0,0), += the others i-major, then / (ss*ss), in float32."""
    acc = samples[0::ss, 0::ss].copy()
    for i in range(ss):
        for j in range(ss):
            if i or j:
                acc = acc + samples[i::ss, j::ss]
    return acc / np.float32(ss * ss)


def box_average(samples, ss):
    """The workaround's host-side average (any order will do for it)."""
    w, h = samples.shape[0] // ss, samples.shape[1] // ss
    return samples.reshape(w, ss, h, ss, 3).mean(axis=(1, 3), dtype=np.float32)


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def cell(s, digits=1):
    return f"{s['median']:.{digits}f} ({s['min']:.{digits}f}..{s['max']:.{digits}f})"


def quiet_scene(name, cam):
    # the library's scene builders print to the C stdout (e.g. SCENE 2's object count): to stderr, out of the report
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        return api.Scene().build(name, cam)
    finally:
        ctypes.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)


class Legs:
    def __init__(self, ctx, flat, camx, p, ss, max_host_bytes):
        self.ctx, self.flat, self.camx, self.p, self.ss = ctx, flat, camx, p, ss
        w, h = p.width, p.height
        self.sp = api.default_params(ss * w, ss * h, p.max_depth)
        self.hb = [api.HostBuffer(w * h * 12) for _ in range(2)]
        self.out = {"float": [b.array(np.float32, (w, h, 3)) for b in self.hb],
                    "rgb8": [b.array(np.uint8, (w, h, 3)) for b in self.hb]}
        sample_bytes = ss * w * ss * h * 12
        self.sample_host = sample_bytes <= max_host_bytes
        self.hs = api.HostBuffer(sample_bytes) if self.sample_host else None
        self.samples = self.hs.array(np.float32, (ss * w, ss * h, 3)) if self.sample_host else None

    def _ss(self, fmt, out):
        if fmt == "float":
            return self.ctx.render_ss(self.p, self.ss, out=out)[1]
        return self.ctx.render_ss_rgb8(self.p, self.ss, out=out)[1]

    def blocking(self, fmt, n):
        rms = []
        t0 = time.perf_counter()
        for _ in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            rms.append(max(self._ss(fmt, self.out[fmt][0]).render_ms))
        return n / (time.perf_counter() - t0), statistics.median(rms)

    def in_flight(self, fmt, n):
        w = self.p.width
        t0 = time.perf_counter()
        tickets = []
        for i in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            out = self.out[fmt][i % 2]
            tickets.append(self.ctx.render_async_ss(self.p, self.ss, 0, w, out) if fmt == "float"
                           else self.ctx.render_async_ss_rgb8(self.p, self.ss, 0, w, out))
            if len(tickets) == 2:
                self.ctx.wait(tickets.pop(0))
        for t in tickets:
            self.ctx.wait(t)
        return n / (time.perf_counter() - t0)

    def sample(self, n, average=False):
        rms = []
        t0 = time.perf_counter()
        for _ in range(n):
            self.ctx.upload_flat(self.flat, self.camx)
            if self.sample_host:
                _, st = self.ctx.render(self.sp, out=self.samples)
                if average:
                    box_average(self.samples, self.ss)
            else:
                st = self.ctx.render_device(self.sp)
            rms.append(max(st.render_ms))
        return n / (time.perf_counter() - t0), statistics.median(rms)


def check(ctx, p, ss, sp):
    """Column ranges of the supersampled frame against resolve() of the plain render of their sample columns."""
    w = p.width
    got, st = ctx.render_ss(p, ss)
    bad = 0
    for c0 in (0, w // 2 - 32, w - 64):
        samples, _ = ctx.render(sp, ss * c0, ss * (c0 + 64))
        want = resolve(samples, ss)
        bad += int((got[c0:c0 + 64].view(np.uint32) != want.view(np.uint32)).any(-1).sum())
    return {"pixels_checked": 3 * 64 * p.height, "pixels_differing": bad, "gpu_launches": st.gpu_launches}


def measure(name, ss, rounds, n_gpus, max_host_bytes):
    scene_name, w, h, d = WORKLOADS[name]
    cam = api.Camera()
    scene = quiet_scene(scene_name, cam)
    flat, camx = scene.flatten(), cam.export()
    p = api.default_params(w, h, d)
    ctx = api.Context([0])
    ctx.upload_flat(flat, camx)
    legs = Legs(ctx, flat, camx, p, ss, max_host_bytes)
    res = {"workload": name, "W": w, "H": h, "depth": d, "ss": ss, "samples_per_frame": ss * ss * w * h,
           "sample_frame_bytes": ss * ss * w * h * 12, "sample_leg_to_host": legs.sample_host,
           "correct": check(ctx, p, ss, legs.sp)}
    for fmt in ("float", "rgb8"):             # warm-up of every call
        legs.blocking(fmt, 2)
        legs.in_flight(fmt, 4)
    legs.sample(2, average=legs.sample_host)
    t0 = time.perf_counter()
    legs.blocking("float", 2)
    frame_s = (time.perf_counter() - t0) / 2
    n = int(min(40, max(4, 0.4 / frame_s)))
    data = {k: [] for k in ("float_blocking", "float_async", "rgb8_blocking", "rgb8_async", "float_render_ms",
                            "rgb8_render_ms", "sample_blocking", "sample_render_ms", "workaround")}
    for r in range(rounds):
        for leg in (("ss", "sample") if r % 2 == 0 else ("sample", "ss")):
            if leg == "ss":
                for fmt in (("float", "rgb8") if r % 2 == 0 else ("rgb8", "float")):
                    fps, rms = legs.blocking(fmt, n)
                    data[f"{fmt}_blocking"].append(fps)
                    data[f"{fmt}_render_ms"].append(rms)
                    data[f"{fmt}_async"].append(legs.in_flight(fmt, n))
            else:
                fps, rms = legs.sample(n)
                data["sample_blocking"].append(fps)
                data["sample_render_ms"].append(rms)
                if legs.sample_host:
                    data["workaround"].append(legs.sample(max(2, n // 4), average=True)[0])
    out = {"frames_per_window": n}
    out.update({k: summary(v) for k, v in data.items() if v})
    out["resolve_ms"] = summary([a - b for a, b in zip(data["float_render_ms"], data["sample_render_ms"])])
    out["resolve_share"] = summary([(a - b) / b for a, b in zip(data["float_render_ms"], data["sample_render_ms"])])
    res["1gpu"] = out
    del legs
    if n_gpus > 1:
        multi = api.Context(list(range(n_gpus)))
        multi.upload_flat(flat, camx)
        for _ in range(8):                        # the multi-device ctx re-cuts after every whole-frame render
            multi.render_ss(p, ss)
        ml = Legs(multi, flat, camx, p, ss, 0)
        res[f"{n_gpus}gpu"] = {"float_blocking": summary([ml.blocking("float", n)[0] for _ in range(rounds)])}
        del ml
        multi.close()
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("workloads", nargs="*", default=DEFAULT_WORKLOADS)
    ap.add_argument("--ss", default="1,2,4", help="samples per axis, comma-separated")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--max-host-gb", type=float, default=2.0, help="largest sample frame copied to host memory")
    ap.add_argument("--json", default=None, help="write the results here as well")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    n_gpus = api.device_count()
    if n_gpus < 1:
        sys.exit("no CUDA device: this tool measures on the GPU and has no CPU path")
    info = {"devices": device_info(), "visible_gpus": n_gpus, "rounds": args.rounds, "results": []}
    print("device (name, power limit, max SM clock):", *info["devices"], sep="\n  ")
    print(f"visible GPUs: {n_gpus}; {args.rounds} rounds, legs alternating; frames/s as median (min..max)")
    if n_gpus < 2:
        print("multi-device legs: not measured (one GPU visible)")
    for name in args.workloads:
        for ss in (int(s) for s in args.ss.split(",")):
            r = measure(name, ss, args.rounds, n_gpus, int(args.max_host_gb * 1e9))
            info["results"].append(r)
            t, c = r["1gpu"], r["correct"]
            gs = r["samples_per_frame"] / 1e9
            print(f"\n== {name} ({r['W']}x{r['H']} d{r['depth']}) ss={ss}: {r['samples_per_frame'] / 1e6:.1f} M samples, "
                  f"sample frame {r['sample_frame_bytes'] / 1e6:.0f} MB")
            print(f"  correct: {c['pixels_differing']} of {c['pixels_checked']} checked pixels differ from resolve() of "
                  f"the sample columns; {c['gpu_launches']} launches per frame")
            for fmt in ("float", "rgb8"):
                b, a = t[f"{fmt}_blocking"], t[f"{fmt}_async"]
                print(f"  ss {fmt:5s}  blocking {cell(b)} f/s = {b['median'] * gs:.2f} Gsamples/s   async {cell(a)} f/s = "
                      f"{a['median'] * gs:.2f} Gsamples/s   render_ms {cell(t[f'{fmt}_render_ms'], 3)}")
            kind = "pinned host" if r["sample_leg_to_host"] else "device only, one launch"
            print(f"  sample ({kind}) blocking {cell(t['sample_blocking'])} f/s   render_ms {cell(t['sample_render_ms'], 3)}")
            print(f"  resolve + scratch: {cell(t['resolve_ms'], 3)} ms = {100 * t['resolve_share']['median']:.1f} % "
                  f"of the sample frame's render_ms")
            if "workaround" in t:
                print(f"  workaround (sample frame to host + numpy average): {cell(t['workaround'], 2)} f/s; "
                      f"ss float blocking is {t['float_blocking']['median'] / t['workaround']['median']:.1f}x")
            else:
                print("  workaround: not measured (sample frame above --max-host-gb)")
            for tag in [k for k in r if k.endswith("gpu") and k != "1gpu"]:
                print(f"  {tag} ss float blocking {cell(r[tag]['float_blocking'])} f/s")
            sys.stdout.flush()
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(info, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
