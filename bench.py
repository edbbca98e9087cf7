#!/usr/bin/env python
"""bench.py — Mrays/s (primary + shadow + reflection) and frames/s of the render path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

One "step" = one frame of the workload.  The default workload is BASELINE.json configs[4]
(synth256_8k_d10: the mirror-heavy 256-sphere scene at 7680x4320, depth 10) — the largest config, it fits
one GPU, and it is the one the north_star's 1 -> 8 GPU target is stated on.  With N ranks (torchrun, one
process per GPU) the frame is split into N cost-balanced column bands, one per rank, with no collective on
the data path (the reference's strategy-1 band partition, RayTracer.cpp:904-906, with the band axis turned
so that a band is one contiguous slice of the x-major pixel array); each rank's band is copied back to its
own pinned host buffer in the e2e leg.  Rank 0 prints ONE JSON line.

  value      rays / kernel time, scene resident in HBM, output left in HBM; CUDA events on the launching
             stream around every launch (tcrt_stats.render_ms), L2 flushed between steps, max over ranks.
  e2e        the same metric through the C-ABI call a user makes with HOST buffers: every step re-uploads
             the flattened scene (H2D) and tcrt_render_columns() copies the finished band into pinned host
             memory (D2H); wall clock around the calls, max over ranks.  e2e_async: the same with two frames in
             flight (tcrt_render_async / tcrt_wait).
  configs    the same two measurements (fewer steps) for ALL FIVE BASELINE configs at this N, each with
             frac_executed / frac_algorithmic and a parity verdict.
  parity     outside the timed region, at every N: every rank compares sampled columns of its finished band
             bit for bit (md5 of the float32 bytes) with columns rendered by the reference itself
             (tests/golden/bench_columns.json, made by tests/golden/make_bench_columns.py from
             oracle/_ref/ref_render).  At N > 1 rank 0 also renders one frame through ONE multi-device
             tcrt_ctx over all N GPUs (the drop-in surface of include/RayTracer.h) and checks the stitched
             frame and its .txt the same way.
  roofline   FP32-pipe bound (SURVEY §8d).  frac = frac_executed: FP32 lane-instructions per second
             (FADD+FMUL+FFMA thread instructions of the committed ncu capture of this kernel on this
             workload, per ray, x this run's rays / this run's kernel time) over the lane-instruction rate
             measured live by tcrt_fp32_peak.  frac_algorithmic: the flops the REFERENCE's linear sweep over
             every object would spend on these rays (oracle counters x SURVEY §8d constants) over the same
             peak — with culling (box clusters, BVH) this is a speed-up over the linear sweep, not a
             fraction of the machine, and may exceed 1.
  cpu_baseline  the reference itself (oracle/_ref/ref_render: calculatePixel & co. compiled from the
             reference's sources) on the host cores, bounded sample; rank 0, N=1 only.
  also       e2e_multiframe (scene resident, new camera per frame, frame to the host), e2e_txt (render + GPU
             "%f" formatting + D2H + file write), bands / kernel_ms_per_rank /
             balance_max_over_mean_per_iteration (the cost-balanced cut and how its feedback converged).

--impl reference times the reference on all host cores (one process per core, column bands — the
reference's own strategy-1 partition), each step a bounded column sample of the workload.  That arm never
imports tilecoderaytracer_b200 and never maps libtcrt.so: the ray count of its sample comes from
oracle/_ref/ref_count (the reference plus two counter increments, run once, never timed).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (which may be read-only)

# name -> (scene, W, H, depth): BASELINE.json configs[0..4] (+ the reference's SCENE 2, + reduced copies)
WORKLOADS = {
    "default_500x504_d50": ("default", 500, 504, 50),      # configs[0], the reference's own case
    "default_1080p_d5": ("default", 1920, 1080, 5),        # configs[1]
    "default_4k_d50": ("default", 3840, 2160, 50),         # configs[2]
    "synth1024_4k_d50": ("synth1024", 3840, 2160, 50),     # configs[3]
    "synth256_8k_d10": ("synth256", 7680, 4320, 10),       # configs[4]  <- default workload at every N
    "two_mirrors_1080p_d50": ("two_mirrors", 1920, 1080, 50),
    # reduced-resolution copies of configs[3], [4] for quick ncu captures (tools/profile_run.py)
    "synth1024_1080p_d50": ("synth1024", 1920, 1080, 50),
    "synth256_1080p_d10": ("synth256", 1920, 1080, 10),
}
BASELINE_CONFIGS = ["default_500x504_d50", "default_1080p_d5", "default_4k_d50", "synth1024_4k_d50", "synth256_8k_d10"]
DEFAULT_WORKLOAD = "synth256_8k_d10"
METRIC = "Mrays/s (primary+shadow+reflection)"
# ncu capture whose per-ray FP32 lane-instruction count stands for a workload (same scene, same depth)
CAPTURE_OF = {"synth256_8k_d10": "synth256_1080p_d10", "synth1024_4k_d50": "synth1024_1080p_d50"}
NCU_METRICS = os.path.join(ROOT, "profiles", "ncu_metrics_r2.json")
GOLDEN_COLUMNS = os.path.join(ROOT, "tests", "golden", "bench_columns.json")
DUMP_BYTES = 48 << 20    # --dump-outputs: pixel bytes at most; with the column indices and counters well under 64 MB


# ---- clocks during the timed region (NVML) ---------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting",
    }

    def __init__(self, index: int, period_s: float = 0.002):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:   # NVML missing: report that, do not invent clocks
            self.nv, self.err = None, repr(e)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": self.err}
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def equal_bands(width: int, n: int):
    """The reference's static partition (strategy 1, RayTracer.cpp:904-906): n equal bands."""
    return [((width * r) // n, (width * (r + 1)) // n) for r in range(n)]


def workload_config(name, n_gpus):
    scene, w, h, depth = WORKLOADS[name]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    how = "" if world > 1 or n_gpus == 1 else " (one process, multi-device tcrt_ctx)"
    return {"workload": name, "scene": scene, "width": w, "height": h, "max_depth": depth, "shadows": True,
            "reflections": True, "partition": f"{n_gpus} cost-balanced column band(s), one per GPU, no collective" + how,
            "l2": "flushed between timed steps (the kernel reads no large input: the scene is a few KB in shared memory, BVH nodes and grid cells a few hundred KB read through L1)"}


# ---- the reference on the host cores (no import of the product anywhere below) -------------------------------
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def ref_processes(scene, w, h, depth, bands, stride, binary="ref_render"):
    """Runs one reference process per band concurrently; returns (max in-loop render seconds, wall seconds,
    pixels, infos)."""
    t0 = time.perf_counter()
    procs = [subprocess.Popen([os.path.join(REF_DIR, binary), scene, str(w), str(h), str(depth), str(x0), str(x1), "-",
                               "--stride", str(stride)], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE,
                              cwd=tempfile.gettempdir()) for x0, x1 in bands if x1 > x0]
    infos = []
    for p in procs:
        err = p.communicate()[1].decode()
        if p.returncode != 0:
            raise RuntimeError(f"{binary} failed: " + err[-300:])
        infos.append(json.loads(err.strip().splitlines()[-1]))
    wall = time.perf_counter() - t0
    return max(i["render_s"] for i in infos), wall, sum(i["pixels"] for i in infos), infos


def ref_rays(scene, w, h, depth, bands, stride):
    """Rays (primary + shadow + reflection) of exactly the pixels ref_processes renders, counted by the
    reference itself (oracle/_ref/ref_count; untimed)."""
    _, _, _, infos = ref_processes(scene, w, h, depth, bands, stride, binary="ref_count")
    return sum(i["rays_primary"] + i["rays_shadow"] + i["rays_reflect"] for i in infos)


def have_reference():
    return all(os.access(os.path.join(REF_DIR, b), os.X_OK) for b in ("ref_render", "ref_count"))


def pick_stride(w, h, us_per_pixel, cores, budget_s):
    """Column stride so that (w/stride)*h pixels on `cores` processes take about budget_s."""
    full_s = w * h * us_per_pixel * 1e-6 / max(1, cores)
    stride = max(1, int(full_s / budget_s + 0.999))
    return min(stride, max(1, w // max(1, cores)))


def calibrate_us_per_pixel(scene, w, h, depth):
    """One thin column sample of the reference (about a second) -> single-thread us/pixel."""
    stride = max(1, w // 12)
    render_s, _, pixels, _ = ref_processes(scene, w, h, depth, [(0, w)], stride)
    return render_s * 1e6 / pixels


def run_reference(args):
    """--impl reference: the reference's CPU implementation on all host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    scene, w, h, depth = WORKLOADS[args.workload]
    if not have_reference():
        emit({"impl": "reference", "unavailable": "oracle/_ref/ref_render not built"})
        return 0
    cores = os.cpu_count() or 1
    procs = min(cores, w)
    us_pp = calibrate_us_per_pixel(scene, w, h, depth)
    total_budget = float(os.environ.get("TCRT_REF_BUDGET_S", "120"))
    stride = pick_stride(w, h, us_pp, procs, total_budget / max(1, args.steps + args.warmup + 1))
    bands = equal_bands(w, procs)
    rays = ref_rays(scene, w, h, depth, bands, stride)
    for _ in range(args.warmup):
        ref_processes(scene, w, h, depth, bands, stride)
    times = []
    pixels = 0
    for _ in range(args.steps):
        render_s, wall, pixels, _ = ref_processes(scene, w, h, depth, bands, stride)
        times.append(render_s)
    t = sum(times)
    mrays = rays * args.steps / t / 1e6
    frac = pixels / float(w * h)
    sample = (f"{procs} processes x equal column bands, every {stride}th column of each band "
              f"({pixels} of {w * h} pixels per step); time = slowest process's pixel loop; rays counted by ref_count")
    line = {
        "impl": "reference", "metric": METRIC, "value": mrays, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, args.gpus), "frames_per_s_equiv": args.steps * frac / t,
        "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": procs, "kind": "reference", "sample": sample,
                         "single_thread_us_per_pixel": us_pp},
        "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def cpu_baseline(scene, w, h, depth):
    """The reference on the host cores, single thread and one process per core, ~6 s each."""
    if not have_reference():
        # the oracle port instead (kind "port"), single thread
        stride = max(1, w // 16)
        t0 = time.perf_counter()
        cnt = oracle_sample(scene, w, h, depth, stride)
        dt = time.perf_counter() - t0
        return {"value": cnt["rays"] / dt / 1e6, "unit": "Mrays/s", "cores": 1, "kind": "port",
                "sample": f"every {stride}th column, oracle/tcrt_oracle.c single thread"}
    cores = os.cpu_count() or 1
    us_pp = calibrate_us_per_pixel(scene, w, h, depth)
    s1 = pick_stride(w, h, us_pp, 1, 6.0)
    r1, _, px1, _ = ref_processes(scene, w, h, depth, [(0, w)], s1)
    c1 = ref_rays(scene, w, h, depth, [(0, w)], s1)
    procs = min(cores, w)
    bands = equal_bands(w, procs)
    sa = pick_stride(w, h, us_pp, procs, 6.0)
    ra, _, pxa, _ = ref_processes(scene, w, h, depth, bands, sa)
    ca = ref_rays(scene, w, h, depth, bands, sa)
    return {
        "value": ca / ra / 1e6, "unit": "Mrays/s", "cores": procs, "kind": "reference",
        "sample": f"{procs} processes (one per host core) x column bands, every {sa}th column ({pxa} of {w * h} pixels); "
                  f"time = slowest process's pixel loop",
        "single_thread": {"value": c1 / r1 / 1e6, "unit": "Mrays/s", "cores": 1,
                          "sample": f"every {s1}th column ({px1} pixels)", "us_per_pixel": r1 * 1e6 / px1},
        "frames_per_s_equiv": (pxa / float(w * h)) / ra,
    }


# ---- helpers of the B200 arm ---------------------------------------------------------------------------------
def oracle_sample(scene_name, w, h, depth, stride):
    """Counters (rays, flops of the reference's linear sweep) of the column sample x = 0, stride, ... from the oracle."""
    from oracle import oracle_py as O
    from tilecoderaytracer_b200 import api

    cam = api.Camera()
    scene = api.Scene().build(scene_name, cam)
    _, cnt = O.render(scene.flatten(), cam.export(), api.default_params(w, h, depth), 0, w, stride)
    cnt["rays"] = cnt["rays_primary"] + cnt["rays_shadow"] + cnt["rays_reflect"]
    return cnt


def ncu_metrics(workload):
    try:
        return json.load(open(NCU_METRICS))[CAPTURE_OF.get(workload, workload)]
    except Exception:
        return None


def measured_hbm_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0   # fallback of B200_PROFILING.md


def scene_bytes(flat):
    n = flat.n_objects
    return 4 * (4 * flat.n_spheres + 16 * flat.n_fin_planes + 16 * flat.n_inf_planes + (4 + 4 + 4 + 8 + 4) * n
                + flat.n_spheres + flat.n_fin_planes + flat.n_inf_planes + flat.n_lights + 8 * flat.n_textures)


def golden_columns(workload):
    try:
        return json.load(open(GOLDEN_COLUMNS))["workloads"][workload]
    except Exception:
        return None


def check_columns(workload, band, x0, x1):
    """(columns checked, columns equal): sampled columns of `band` (= columns [x0, x1) of the frame, host
    float32 [x1-x0, H, 3]) against the reference's own render."""
    g = golden_columns(workload)
    if g is None:
        return 0, 0
    n = ok = 0
    for c, want in zip(g["columns"], g["md5"]):
        if x0 <= c < x1:
            n += 1
            ok += hashlib.md5(band[c - x0].tobytes()).hexdigest() == want
    return n, ok


class Dist:
    """torch.distributed plumbing of one run: NCCL for the reductions next to the GPU work, a gloo group for
    host-side waits (a rank parked in an NCCL barrier would spin on its GPU)."""

    def __init__(self, args):
        from tilecoderaytracer_b200 import distributed as D

        self.D = D
        self.rank, self.world, self.local = D.env_world()
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        self.tdev = None
        self.cpu_group = None
        if self.world > 1:
            import torch
            import torch.distributed as dist

            torch.cuda.set_device(self.local)
            self.tdev = torch.device("cuda", self.local)
            D.init("nccl")
            self.cpu_group = dist.new_group(backend="gloo")

    def barrier(self):
        if self.world > 1:
            import torch

            self.D.barrier()
            torch.cuda.synchronize()

    def host_barrier(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier(group=self.cpu_group)

    def max(self, v):
        return self.D.reduce_max(v, self.tdev)

    def sum(self, v):
        return self.D.reduce_sum(v, self.tdev)

    def min(self, v):
        return -self.D.reduce_max(-v, self.tdev)

    def gather(self, v):
        return self.D.gather_floats(v, self.tdev)

    def gather_objects(self, obj):
        """Every rank's object on rank 0, in rank order (None on the other ranks); over gloo, outside timed regions."""
        if self.world == 1:
            return [obj]
        import torch.distributed as dist

        out = [None] * self.world if self.rank == 0 else None
        dist.gather_object(obj, out, dst=0, group=self.cpu_group)
        return out

    def bcast(self, obj):
        return self.D.broadcast_object(obj)


def dump_outputs(ctx, dist, out_dir, params, x0, x1, st):
    """--dump-outputs: what the last timed step computed, as its caller receives it: the band tcrt_render_device left
    on the device (fetched with tcrt_download) and the ray counters of its tcrt_stats.  A frame larger than DUMP_BYTES
    is sampled by whole columns whose x positions come from a fixed seed, so two runs with the same arguments (and two
    builds of the project) write the same pixels.
      image.npy          float32 [columns, height, 3]: the sampled columns, x-major like the frame
      image_columns.npy  float64 [columns]: the x of each of them
      rays.npy           float64 [3]: primary, shadow and reflection rays of the whole frame"""
    import numpy as np

    w, h = params.width, params.height
    band = ctx.download(np.empty((x1 - x0, h, 3), np.float32))
    k = min(w, DUMP_BYTES // (h * 3 * 4))
    cols = np.arange(w) if k == w else np.sort(np.random.default_rng(0).choice(w, k, replace=False))
    parts = dist.gather_objects(band[cols[(cols >= x0) & (cols < x1)] - x0])
    rays = [dist.sum(v) for v in (st.rays_primary, st.rays_shadow, st.rays_reflect)]
    if dist.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "image.npy"), np.concatenate(parts, 0))
        np.save(os.path.join(out_dir, "image_columns.npy"), cols.astype(np.float64))
        np.save(os.path.join(out_dir, "rays.npy"), np.array(rays, np.float64))


def run_workload(ctx, dist, args, name, steps, warmup, inproc, sample_clocks=False, host=None, dump_dir=None):
    """Kernel-only and end-to-end measurement of one workload at this N, plus its parity verdict."""
    import numpy as np

    from tilecoderaytracer_b200 import api
    from tilecoderaytracer_b200.partition import rebalance

    rank, world = dist.rank, dist.world
    scene_name, w, h, depth = WORKLOADS[name]
    cam = api.Camera()
    scene = api.Scene().build(scene_name, cam)
    params = api.default_params(w, h, depth)
    ctx.upload(scene, cam)
    flat, camx = scene.flatten(), cam.export()
    # one column band per rank; the cut is cost-balanced (a low-resolution pre-pass on rank 0 that counts
    # bounces per column, shared once at setup) and outside the timed region
    bands = ctx.balance_columns(params, world) if rank == 0 else None
    bands = dist.bcast(bands)
    if inproc:
        for _ in range(12):                   # the multi-device ctx re-cuts after every whole-frame render
            ctx.render_device(params)
    # ---- at N > 1, feedback on the cut: every rank re-cuts from the same gathered band times (so all agree)
    # until the slowest band is within 1 % of the mean; the cut is then frozen ---------------------------------
    balance_log = []
    if world > 1:
        for _ in range(16):
            x0, x1 = bands[rank]
            ms = min(ctx.render_device(params, x0, x1).render_ms[0] for _ in range(2)) if x1 > x0 else 0.0
            all_ms = dist.gather(ms)
            balance_log.append(max(all_ms) / (sum(all_ms) / world))
            if balance_log[-1] < 1.01:
                break
            new = rebalance(bands, all_ms, w)
            if any(b[1] - b[0] < 4 for b in new):      # decided from the shared list: every rank stops together
                break
            bands = new
    x0, x1 = bands[rank]
    for _ in range(max(3, warmup)):
        st = ctx.render_device(params, x0, x1)
    # ---- timed: K launches, CUDA events around each, L2 flushed in between ------------------------------------
    dist.barrier()
    kernel_ms, rays_rank, launches = [], 0, 0
    wall0 = time.perf_counter()
    with ClockSampler(dist.local) as clocks:
        for _ in range(steps):
            ctx.flush_l2()
            st = ctx.render_device(params, x0, x1)
            kernel_ms.append(max(st.render_ms))       # in-process multi-device: the slowest device
            rays_rank = st.rays
            launches += st.gpu_launches
    wall = time.perf_counter() - wall0
    dist.barrier()
    if dump_dir is not None:
        dump_outputs(ctx, dist, dump_dir, params, x0, x1, st)
    t_rank_ms = sum(kernel_ms)
    t_ms = dist.max(t_rank_ms)                         # slowest rank, device time
    rank_ms = [t / steps for t in dist.gather(t_rank_ms)]
    if inproc:
        rank_ms, bands = list(st.render_ms), st.bands
    rays_total = dist.sum(rays_rank)                   # per frame
    res = {
        "workload": name, "ms": t_ms / steps, "mrays_s": rays_total * steps / (t_ms * 1e-3) / 1e6,
        "frames_s": steps / (t_ms * 1e-3), "rays_per_frame": int(rays_total), "steps": steps,
        "gpu_launches": int(dist.sum(launches)), "bands": [list(b) for b in bands], "kernel_ms_per_rank": rank_ms,
        "balance_max_over_mean_per_iteration": balance_log, "wall_ms_per_step_incl_flush": 1e3 * wall / steps,
        "kernel_ms_rank_mean": statistics.mean(kernel_ms), "rays_rank": rays_rank,
    }
    if sample_clocks:
        res["clocks"] = clocks.summary()

    # ---- e2e: host buffers, H2D scene + D2H band inside the timed region ----------------------------------------
    # `e2e`: every step re-sends the flattened scene (tcrt_upload_scene) and renders into pinned host memory with
    # the blocking call (tcrt_render_columns), one frame at a time.  `e2e_async`: the call sequence of a user who
    # streams frames — the frame is queued with tcrt_render_async into one of two pinned buffers and the previous
    # frame is waited for (tcrt_wait) while this one renders.
    ex0, ex1 = (0, w) if inproc else (x0, x1)
    band_floats = (ex1 - ex0) * h * 3
    if host is None or host[0].nbytes < band_floats * 4:
        host = [api.HostBuffer(band_floats * 4) for _ in range(2)]
    outs = [hb.array(np.float32, (ex1 - ex0, h, 3)) for hb in host]
    out = outs[0]
    e2e_steps = max(3, min(steps, 30))
    for _ in range(2):
        ctx.upload_flat(flat, camx)
        ctx.render(params, ex0, ex1, out)
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.upload_flat(flat, camx)
        ctx.render(params, ex0, ex1, out)
    sync_s = dist.max(time.perf_counter() - t0)
    dist.barrier()
    t0 = time.perf_counter()
    tickets = []
    for i in range(e2e_steps):
        ctx.upload_flat(flat, camx)
        tickets.append(ctx.render_async(params, ex0, ex1, out=outs[i % 2]))
        if len(tickets) == 2:
            ctx.wait(tickets.pop(0))
    for t in tickets:
        ctx.wait(t)
    e2e_s = dist.max(time.perf_counter() - t0)
    out = outs[(e2e_steps - 1) % 2]
    res["e2e"] = {"value": rays_total * e2e_steps / sync_s / 1e6, "unit": "Mrays/s",
                  "h2d_bytes_per_step": int(scene_bytes(flat) + 64), "d2h_bytes_per_step": int(band_floats * 4 + 32),
                  "frames_per_s": e2e_steps / sync_s, "steps": e2e_steps,
                  "what": "per frame: tcrt_upload_scene + tcrt_render_columns (blocking) into pinned host memory, wall clock"}
    res["e2e_async"] = {"value": rays_total * e2e_steps / e2e_s / 1e6, "unit": "Mrays/s", "frames_per_s": e2e_steps / e2e_s,
                        "h2d_bytes_per_step": int(scene_bytes(flat) + 64), "d2h_bytes_per_step": int(band_floats * 4 + 32),
                        "what": "per frame: tcrt_upload_scene + tcrt_render_async into one of two pinned host buffers, tcrt_wait for "
                                "the previous frame (two frames in flight); wall clock over all frames incl. the last wait"}
    if name in ("default_1080p_d5", args.workload) and not inproc:
        # ---- multi-frame mode (SURVEY §8f): scene resident, a new camera per frame, frame to the host ----------
        import copy

        n_mf = max(6, min(steps * 2, 60))
        cams = []
        for i in range(n_mf):
            c = copy.copy(camx)
            c.eye[0] = camx.eye[0] + 0.002 * i       # a slow dolly: every frame is a different image
            cams.append(c)
        dist.barrier()
        t0 = time.perf_counter()
        tickets = []
        for i, c in enumerate(cams):
            ctx.set_camera(c)
            tickets.append(ctx.render_async(params, ex0, ex1, out=outs[i % 2]))
            if len(tickets) == 2:
                ctx.wait(tickets.pop(0))
        for t in tickets:
            ctx.wait(t)
        mf_s = dist.max(time.perf_counter() - t0)
        ctx.set_camera(camx)
        res["e2e_multiframe"] = {"frames_per_s": n_mf / mf_s, "frames": n_mf,
                                 "what": "tcrt_set_camera + tcrt_render_async into pinned host memory per frame, two frames in "
                                         "flight; scene stays on the device"}
        ctx.render(params, ex0, ex1, out)           # the frame the parity check below looks at
    # ---- parity of what the e2e leg left in host memory, against the reference's own columns ---------------------
    n, ok = check_columns(name, out, ex0, ex1)
    n_all, ok_all = int(dist.sum(n)), int(dist.sum(ok))
    res["parity"] = {"checked": n_all > 0, "ok": n_all > 0 and ok_all == n_all, "columns": n_all, "columns_equal": ok_all,
                     "against": "tests/golden/bench_columns.json: md5 of float32 columns rendered by the reference itself "
                                "(oracle/_ref/ref_render); every rank checks the columns inside its own band"}
    res["_ctx_state"] = (params, x0, x1, out, flat, camx, host)
    return res


def _num(v):
    """Leading number of an exported ncu value ("78.03 %" -> 78.03); None when absent."""
    if v is None:
        return None
    try:
        return float(str(v).split()[0].replace(",", ""))
    except ValueError:
        return None


def fractions(name, res, peak):
    """frac_executed / frac_algorithmic of one measured workload (rank 0)."""
    scene_name, w, h, depth = WORKLOADS[name]
    kernel_s = res["kernel_ms_rank_mean"] * 1e-3
    out = {"frac_executed": None, "frac_algorithmic": None}
    m = ncu_metrics(name)
    if m and m.get("fp32_lane_inst_per_ray"):
        out["fp32_lane_inst_per_ray"] = m["fp32_lane_inst_per_ray"]
        out["executed_tera_inst_s"] = m["fp32_lane_inst_per_ray"] * res["rays_rank"] / kernel_s / 1e12
        out["frac_executed"] = out["executed_tera_inst_s"] / peak["unfused_tera_inst"]
        out["capture"] = m.get("capture")
    cnt = oracle_sample(scene_name, w, h, depth, max(1, w // 24))
    fpr = cnt["flops"] / cnt["rays"]
    out["algorithmic_flops_per_ray"] = fpr
    out["algorithmic_tflops"] = fpr * res["rays_rank"] / kernel_s / 1e12
    out["frac_algorithmic"] = out["algorithmic_tflops"] / peak["unfused_tera_inst"]
    return out


def multi_device_check(world):
    """Rank 0, outside every timed region: ONE tcrt_ctx over all GPUs of the box (the in-process band split the
    drop-in raytrace_main(..., devices) uses) renders default_4k_d50; the stitched frame's sampled columns and
    the md5 of its .txt pixel lines must equal the reference's."""
    import numpy as np

    from tilecoderaytracer_b200 import api

    name = "default_4k_d50"
    scene_name, w, h, depth = WORKLOADS[name]
    cam = api.Camera()
    scene = api.Scene().build(scene_name, cam)
    params = api.default_params(w, h, depth)
    ctx = api.Context(list(range(world)))
    try:
        ctx.upload(scene, cam)
        for _ in range(4):
            ctx.render_device(params)
        img, st = ctx.render(params)
        n, ok = check_columns(name, img, 0, w)
        # (no timings here: the other ranks' processes still hold contexts on their GPUs, which this process time-shares)
        out = {"devices": world, "workload": name, "bands": [list(b) for b in st.bands],
               "columns": n, "columns_equal": ok, "ok": n > 0 and n == ok}
        try:
            want = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))["md5"]["default_3840x2160_d50"]
            with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
                path = os.path.join(td, "raytracer_screen.txt")
                ctx.render_device(params)
                ctx.write_txt(params, path, 0.0)
                md5 = hashlib.md5()
                with open(path, "rb") as f:
                    data = f.read()
                body = data[data.index(b"("):]
                md5.update(body)
                out["txt_md5_ok"] = md5.hexdigest() == want["pixel_md5"] and len(body) == want["pixel_bytes"]
                out["ok"] = out["ok"] and out["txt_md5_ok"]
        except KeyError:
            out["txt_md5_ok"] = None
        return out
    finally:
        ctx.close()


def txt_leg(ctx, dist, name, frames=3):
    """render + .txt file of the reference's format (RayTracer.cpp:1574-1626) in tmpfs, at this N.  One rank: the
    whole frame through tcrt_write_txt.  N ranks: rank 0 creates the file (tcrt_txt_create), every rank renders its
    band and writes its lines at their place (tcrt_write_txt_band) — no gather.  The md5 of the pixel lines is
    compared with the reference program's where tests/golden/golden.json has one."""
    from tilecoderaytracer_b200 import api

    rank, world = dist.rank, dist.world
    scene_name, w, h, depth = WORKLOADS[name]
    cam = api.Camera()
    scene = api.Scene().build(scene_name, cam)
    params = api.default_params(w, h, depth)
    ctx.upload(scene, cam)
    bands = dist.bcast(ctx.balance_columns(params, world) if rank == 0 else None)
    x0, x1 = bands[rank]
    td = dist.bcast(tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) if rank == 0 else None)
    path = os.path.join(td, "raytracer_screen.txt")
    times = []
    for i in range(frames + 1):
        dist.host_barrier()
        t0 = time.perf_counter()
        if world == 1:
            ctx.render_device(params)
            ctx.write_txt(params, path, 0.0)
        else:
            if rank == 0:
                api.txt_create(params, path, 0.0)
            dist.host_barrier()
            ctx.render_device(params, x0, x1)
            ctx.write_txt_band(params, path, 0.0)
        dist.host_barrier()
        if i > 0:
            times.append(time.perf_counter() - t0)
    out = None
    if rank == 0:
        size = os.path.getsize(path)
        s = statistics.mean(times)
        out = {"workload": name, "frames_per_s": 1.0 / s, "ms_per_frame": 1e3 * s, "file_bytes": size, "gb_per_s": size / s / 1e9,
               "what": "render + GPU %f formatting + D2H of text + copies into the file (tmpfs), pipelined in 7.9 MB chunks; "
                       + ("tcrt_write_txt" if world == 1 else "tcrt_txt_create on rank 0 + tcrt_write_txt_band on every rank")}
        key = {"default_4k_d50": "default_3840x2160_d50", "default_1080p_d5": "default_1920x1080_d5"}.get(name)
        if key:
            want = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))["md5"][key]
            data = open(path, "rb").read()
            body = data[data.index(b"("):]
            out["md5_equals_reference_file"] = hashlib.md5(body).hexdigest() == want["pixel_md5"] and len(body) == want["pixel_bytes"]
        os.unlink(path)
        os.rmdir(td)
    dist.host_barrier()
    return out


def file_copy_bound(nbytes, threads=8):
    """What the file system allows: `threads` threads copying nbytes from memory into the mapping of a NEW file
    in the same tmpfs (page allocation + copy), GB/s — the .txt leg cannot be faster than this plus the render."""
    import numpy as np

    d = "/dev/shm" if os.path.isdir("/dev/shm") else None
    src = np.ones(nbytes, dtype=np.uint8)
    best = None
    for _ in range(3):
        with tempfile.NamedTemporaryFile(dir=d) as f:
            t0 = time.perf_counter()
            f.truncate(nbytes)
            mm = np.memmap(f.name, dtype=np.uint8, mode="r+", shape=(nbytes,))
            cuts = [nbytes * i // threads for i in range(threads + 1)]
            ts = [threading.Thread(target=lambda a, b: mm.__setitem__(slice(a, b), src[a:b]), args=(cuts[i], cuts[i + 1]))
                  for i in range(threads)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
            dt = time.perf_counter() - t0
            del mm
        best = dt if best is None else min(best, dt)
    return {"bytes": nbytes, "threads": threads, "ms": 1e3 * best, "gb_per_s": nbytes / best / 1e9,
            "what": "numpy slices copied by threads into np.memmap of a new /dev/shm file (page faults + copy), best of 3"}


# ---- the B200 arm -----------------------------------------------------------------------------------------
def run_ours(args):
    from tilecoderaytracer_b200 import api

    dist = Dist(args)
    rank, world, local = dist.rank, dist.world, dist.local
    # --gpus N without torchrun: ONE process drives N GPUs through a multi-device tcrt_ctx (the library
    # cuts, balances and stitches the bands itself); under torchrun: one rank per GPU.
    inproc = world == 1 and args.gpus > 1
    ctx = api.Context(list(range(args.gpus)) if inproc else [local])
    t_start = time.perf_counter()

    head = run_workload(ctx, dist, args, args.workload, args.steps, args.warmup, inproc, sample_clocks=True,
                        dump_dir=args.dump_outputs)
    params, x0, x1, out, flat, camx, hb = head.pop("_ctx_state")
    scene_name, w, h, depth = WORKLOADS[args.workload]
    line = {
        "metric": METRIC, "value": head["mrays_s"], "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": head["ms"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, args.gpus),
        "frames_per_s": head["frames_s"], "rays_per_frame": head["rays_per_frame"],
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
        "wall_ms_per_step_incl_flush": head["wall_ms_per_step_incl_flush"],
        "bands": head["bands"], "kernel_ms_per_rank": head["kernel_ms_per_rank"],
        "balance_max_over_mean_per_iteration": head["balance_max_over_mean_per_iteration"],
        "parity": head["parity"],
        "note": "strong scaling: the frame is fixed and split into N column bands, one per GPU; no collective on the "
                "data path (torch.distributed carries only the barrier and the timing reductions)",
    }

    if "e2e_multiframe" in head:
        line["e2e_multiframe"] = head["e2e_multiframe"]
    line["e2e_async"] = head["e2e_async"]
    # ---- all five BASELINE configs at this N ----------------------------------------------------------------------
    peak = ctx.fp32_peak() if rank == 0 else None
    results = {args.workload: head}
    if not args.quick:
        for name in BASELINE_CONFIGS:
            if name not in results:
                r = run_workload(ctx, dist, args, name, max(3, min(args.steps, 10)), 3, inproc, host=hb)
                if "e2e_multiframe" in r and name == "default_1080p_d5":
                    line["e2e_multiframe_1080p"] = r["e2e_multiframe"]
                r.pop("_ctx_state")
                results[name] = r
    if not args.quick and not inproc:
        txt = {}
        for name in dict.fromkeys(["default_4k_d50", args.workload]):
            txt[name] = txt_leg(ctx, dist, name)
        if rank == 0:
            line["e2e_txt"] = txt[args.workload]
            line["e2e_txt_4k"] = txt["default_4k_d50"]
            line["file_copy_bound"] = file_copy_bound(txt["default_4k_d50"]["file_bytes"])
    if rank == 0:
        cfgs = {}
        for name, r in results.items():
            f = fractions(name, r, peak)
            cfgs[name] = {"ms": r["ms"], "mrays_s": r["mrays_s"], "frames_s": r["frames_s"], "steps": r["steps"],
                          "e2e": {k: r["e2e"][k] for k in ("value", "frames_per_s", "h2d_bytes_per_step", "d2h_bytes_per_step")},
                          "e2e_async": {k: r["e2e_async"][k] for k in ("value", "frames_per_s")},
                          "frac_executed": f["frac_executed"], "frac_algorithmic": f["frac_algorithmic"],
                          "parity_ok": r["parity"]["ok"], "parity_columns": r["parity"]["columns"],
                          "bands": r["bands"], "kernel_ms_per_rank": r["kernel_ms_per_rank"]}
            if name == args.workload:
                fh = f
        line["configs"] = cfgs
        line["parity"]["all_configs_ok"] = all(c["parity_ok"] for c in cfgs.values())
        # ---- roofline of the headline kernel ------------------------------------------------------------------------
        m = ncu_metrics(args.workload) or {}
        kernel_s = head["kernel_ms_rank_mean"] * 1e-3
        band_bytes = (x1 - x0) * h * 12
        line["roofline"] = {
            "bound": "fp32_pipe", "unit": "T lane-inst/s (1 flop each: parity-exact code cannot use FFMA)",
            "achieved": fh.get("executed_tera_inst_s"), "peak": peak["unfused_tera_inst"], "frac": fh["frac_executed"],
            "frac_executed": fh["frac_executed"], "frac_algorithmic": fh["frac_algorithmic"],
            "achieved_algorithmic_tflops": fh["algorithmic_tflops"], "algorithmic_flops_per_ray": fh["algorithmic_flops_per_ray"],
            "fp32_lane_inst_per_ray": fh.get("fp32_lane_inst_per_ray"), "capture": fh.get("capture"),
            "traffic": m.get("dram_bytes_per_launch"),
            "kernel": m.get("kernel", "render_pool_kernel / render_kernel"), "kernel_ms": 1e3 * kernel_s,
            "peak_source": "measured live: tcrt_fp32_peak, dependent FMUL+FADD chains; MEASURED_PEAKS.json has no FP32-pipe figure",
            "peak_fma_tera_inst": peak["fma_tera_inst"],
            "what": "frac = frac_executed = FP32 lane-instructions/s (FADD+FMUL+FFMA thread instructions per ray of the committed "
                    "ncu capture named in `capture`, x this run's rays / this run's kernel time) / peak.  frac_algorithmic = flops of the "
                    "reference's linear sweep over every object for these rays / the same peak: a speed-up over the linear sweep "
                    "(BVH and box clusters skip most of it), not a fraction of the machine",
            # what the FP32 fraction leaves out: how busy the issue ports are and how many lanes an instruction carries
            # (same committed capture; a divergent kernel is bound by these, not by the FP32 pipe)
            "capture_issue_slot_pct": _num(m.get("smsp__issue_active.avg.pct_of_peak_sustained_active")),
            "capture_threads_per_inst": _num(m.get("smsp__thread_inst_executed_per_inst_executed.ratio")),
            "capture_fma_pipe_inst_pct": _num(m.get("sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active")),
            "capture_icache_hit_pct": _num(m.get("sm__icc_request_hit_rate.pct")),
            "hbm_algorithmic_bytes_per_launch": band_bytes,
            "hbm_frac_of_measured": (band_bytes / kernel_s / 1e9) / measured_hbm_gbs(),
        }
    # ---- N > 1: one multi-device ctx over all GPUs, checked against the reference (rank 0; the others wait on the host)
    if world > 1 and not args.quick:
        dist.barrier()
        if rank == 0:
            try:
                line["multi_device_ctx"] = multi_device_check(world)
            except Exception as e:   # reported, not hidden
                line["multi_device_ctx"] = {"ok": False, "error": repr(e)[:300]}
        dist.host_barrier()
    if rank == 0:
        # ---- CPU baseline: the reference itself, bounded sample, N=1 only ---------------------------------------
        if world == 1 and not inproc and not args.no_cpu_baseline and not args.quick:
            line["cpu_baseline"] = cpu_baseline(scene_name, w, h, depth)
        line["bench_wall_s"] = time.perf_counter() - t_start
        emit(line)
    ctx.close()
    dist.D.shutdown()
    return 0


def wait_for_build(paths, timeout_s=600.0):
    """Ranks other than local rank 0 wait until the libraries exist and have stopped growing."""
    t0 = time.time()
    last = None
    while time.time() - t0 < timeout_s:
        if all(os.path.exists(p) for p in paths):
            sizes = [os.path.getsize(p) for p in paths]
            if sizes == last and all(time.time() - os.path.getmtime(p) > 1.0 for p in paths):
                return
            last = sizes
        time.sleep(0.5)
    raise SystemExit("timed out waiting for local rank 0 to build " + ", ".join(paths))


_RESULT_FD = None


def emit(line):
    """The one JSON line of the contract, on the process's original stdout."""
    text = json.dumps(line) + "\n"
    if _RESULT_FD is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, text.encode())


def quiet_stdout():
    """Point fd 1 at stderr for the rest of the run (NCCL prints its version banner to stdout from C, build steps
    chat): stdout then carries the JSON line and nothing else."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline workload only (developer loop)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step (a seeded column sample when large) and its ray "
                         "counters to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 path computed; --impl reference has no such frame")
    quiet_stdout()
    if args.impl == "reference":
        # the prebuilt oracle/_ref travels with the repo; built here only where /root/reference exists
        if int(os.environ.get("RANK", "0")) == 0 and not have_reference() and os.path.isdir("/root/reference"):
            subprocess.run(["bash", os.path.join(ROOT, "oracle", "build_ref.sh")], check=False)
        return run_reference(args)
    from tilecoderaytracer_b200 import build as B

    # the prebuilt in-tree libraries travel with the repo; only a missing one is built here, by local rank 0,
    # while the other ranks wait for the finished files
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        if not os.path.exists(B.LIB_PATH):
            B.build_lib()
        if not os.path.exists(B.ORACLE_LIB_PATH):
            B.build_oracle()
        B.build_ref()
    else:
        wait_for_build([B.LIB_PATH, B.ORACLE_LIB_PATH])
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
