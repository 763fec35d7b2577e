#!/usr/bin/env python
"""bench.py -- Mpaths/s (and Mrays/s) of the hw5 path tracer hot path, one BASELINE.json configuration per run.

  --config 1  practice5_1          (primitives + Monte Carlo lighting) at the scene's own 1024x768, 64 spp;
                                    the reference arm is the reference's own CLI on the whole frame
  --config 2  practice5_dragon_10k        512x512, 128 spp
  --config 3  practice5_dragon_100k       512x512, 128 spp            <- default, the headline
  --config 4  practice5_dragon_100k_glass 512x512, 128 spp
  --config 5  practice5_dragon_100k_metal re-rendered at 3840x2160, 1024 spp

One "step" = one full Scene::Render pass of the scene (W x H x SAMPLES camera paths, RAY_DEPTH 6) spp-sharded over
the N ranks (each rank renders SAMPLES/N samples per pixel with disjoint Philox streams; the float accumulation
buffers are summed onto rank 0 with an NCCL reduce), so scaling is STRONG: the total work per step is fixed.

  value        device-resident throughput: scene already in HBM, timed region = render kernels (+ the NCCL reduce for
               N > 1), CUDA events, max over ranks.
  e2e          the same metric through the C-ABI with host buffers: every step uploads the flattened scene from pinned
               host memory (H2D), renders, resolves to 8-bit and copies the image back (D2H); frames are queued two deep
               (rtc_frame_begin / rtc_frame_end), every frame complete inside the timed region.
  roofline     the dominant kernel against the roof that bounds it; `rooflines` holds all three kernels:
               k_traverse against the measured L2 gather rate (tools/peaks, run live on the same GPU) and the measured
               warp-instruction issue rate, k_shade / k_generate against the measured HBM copy rate.
  cpu_baseline the UNMODIFIED reference on the host cores (oracle/_ref): its CLI on the whole frame for config 1, its
               Scene::Sample loop on a bounded sample of the frame for the dragon scenes.
  load_s, cli_s  scene file -> HBM (parse, both BVH builds, upload), and the wall time of run.sh on the scene.

`--impl reference` times the reference arm as its own JSON line.

`--dump-outputs DIR` writes what the last device-resident timed step computed, the float32 radiance sums over its
samples that render_accumulate leaves in the caller's buffer, as DIR/radiance_sum.npy (H x W x 3).  A frame larger
than 2,097,152 pixels is stored as a fixed, seeded sample of that many pixels: DIR/radiance_sum.npy (n x 3) and the
flat pixel indices it came from, DIR/radiance_sum_pixel.npy (float64).  Seeds depend on the step number only, so two
runs with the same arguments render the same paths and agree up to float summation order.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "Mpaths/s"
CONFIGS = {
    1: {"scene": "practice5_1", "ref": "cli"},
    2: {"scene": "practice5_dragon_10k"},
    3: {"scene": "practice5_dragon_100k"},
    4: {"scene": "practice5_dragon_100k_glass"},
    5: {"scene": "practice5_dragon_100k_metal", "width": 3840, "height": 2160, "spp": 1024},
}
DUMP_PIXELS = 1 << 21   # --dump-outputs: at most 24 MB of sums + 16 MB of pixel indices


def scene_file(name):
    p = os.path.join(ROOT, "scenes", name + ".txt")
    if not os.path.exists(p):
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_scenes.py")])
    return p


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback"


def live_peaks(device):
    """tools/peaks: L2-resident random 96-byte gather (GB/s) and warp-instruction issue rates, measured on the GPU that
    is being benchmarked; the committed copy of an earlier run (profiles/r02_peaks.json) if the library is missing."""
    so = os.path.join(ROOT, "tools", "peaks", "libpeaks.so")
    keys = ["l2_gather96_gbs", "l2_chase96_gbs", "l2_chase96_ns_per_fetch", "ffma_gwinst_s", "alu_gwinst_s",
            "mixed_gwinst_s", "unused", "copy_gbs", "sms", "fp32_tflops"]
    try:
        lib = ctypes.CDLL(so)
        lib.rtc_peaks_measure.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.POINTER(ctypes.c_double)]
        out = (ctypes.c_double * 10)()
        if lib.rtc_peaks_measure(device, 36.0, out) == 0:
            d = dict(zip(keys, [float(v) for v in out]))
            d.pop("unused", None)
            d["source"] = "measured live (tools/peaks)"
            return d
    except OSError:
        pass
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_peaks.json")))
        d["source"] = "profiles/r02_peaks.json (an earlier run on this pool)"
        return d
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith("nvmlClocksThrottleReason") or n.startswith("nvmlClocksEventReason"):
                v = getattr(nv, n)
                if isinstance(v, int) and v:
                    names.setdefault(v, n.replace("nvmlClocksThrottleReason", "").replace("nvmlClocksEventReason", ""))
        while not self.stop_flag.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit and bit & (bit - 1) == 0:
                        self.reasons.add(nm)
            except Exception:
                pass
            self.stop_flag.wait(0.01)

    def result(self):
        self.stop_flag.set()
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        reasons = sorted(r for r in self.reasons if r not in ("GpuIdle", "None", "ApplicationsClocksSetting"))
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.samples)}


def dump_outputs(out_dir, accum, width, height):
    """Writes the float32 accumulation buffer `accum` (a device tensor of H * W * 3 sums) under out_dir, sampled
    to DUMP_PIXELS seeded pixels when the frame is larger."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    npix = width * height
    rgb = accum.view(npix, 3)
    if npix <= DUMP_PIXELS:
        np.save(os.path.join(out_dir, "radiance_sum.npy"), rgb.view(height, width, 3).cpu().numpy())
        return
    pick = np.sort(np.random.default_rng(0).choice(npix, DUMP_PIXELS, replace=False))
    sample = rgb.index_select(0, torch.from_numpy(pick).to(accum.device))
    np.save(os.path.join(out_dir, "radiance_sum.npy"), sample.cpu().numpy())
    np.save(os.path.join(out_dir, "radiance_sum_pixel.npy"), pick.astype(np.float64))


def resolve_config(args):
    cfg = dict(CONFIGS[args.config])
    if args.scene:
        cfg = {"scene": args.scene}
    for k in ("width", "height", "spp"):
        v = getattr(args, k)
        if v > 0:
            cfg[k] = v
    return cfg


def reference_arm(args, rank):
    """The reference's own CPU implementation of the path on the host cores."""
    if rank != 0:
        return 0
    import orclib
    cfg = resolve_config(args)
    cores = os.cpu_count() or 1
    path = scene_file(cfg["scene"])
    steps = args.steps if args.impl == "reference" else 1
    warm = args.warmup if args.impl == "reference" else 0
    if cfg.get("ref") == "cli" and orclib.have_ref() and not any(k in cfg for k in ("width", "height", "spp")):
        # config 1: the reference's own command line on the whole frame (load + render + PPM, as run.sh does)
        exe = os.path.join(ROOT, "oracle", "_ref", "raytracing_hw5")
        s = orclib.Scene(orclib.ref(), path)
        full = (s.width, s.height, s.samples)
        depth = s.ray_depth
        s.close()

        def one():
            with tempfile.TemporaryDirectory() as tmp:
                t0 = time.perf_counter()
                subprocess.run([exe, path, os.path.join(tmp, "out.ppm")], check=True, stdout=subprocess.DEVNULL,
                               stderr=subprocess.DEVNULL, env=dict(os.environ, OMP_NUM_THREADS=str(cores)))
                return time.perf_counter() - t0
        kind, paths = "reference", full[0] * full[1] * full[2]
        sample = "%s, the whole %dx%d, %d spp frame through the reference's CLI (depth %d, %d paths/step)" % (
            cfg["scene"], full[0], full[1], full[2], depth, paths)
    else:
        if not orclib.have_ref():
            backend, kind = orclib.oracle(), "port"   # the reference did not compile here -> the oracle port
        else:
            backend, kind = orclib.ref(), "reference"
        s = orclib.Scene(backend, path)
        full = (cfg.get("width", s.width), cfg.get("height", s.height), cfg.get("spp", s.samples))
        w, h, spp = args.ref_width, args.ref_height, args.ref_spp
        s.override(w, h, spp)
        depth = s.ray_depth

        def one():
            t0 = time.perf_counter()
            if kind == "reference":
                s.ref_render_linear(nthreads=cores)
            else:
                s.render_sum(1, 0, spp, nthreads=cores)
            return time.perf_counter() - t0
        paths = w * h * spp
        sample = "%s at %dx%d, %d spp, depth %d (%d paths/step) of the %dx%d, %d spp frame" % (
            cfg["scene"], w, h, spp, depth, paths, full[0], full[1], full[2])
    for _ in range(warm):
        one()
    times = [one() for _ in range(steps)]
    value = paths / (sum(times) / len(times)) / 1e6
    base = {"value": value, "unit": METRIC, "cores": cores, "kind": kind, "sample": sample}
    if args.impl != "reference":
        return base
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["scene"], "baseline_config": args.config, "width": full[0], "height": full[1],
                       "spp": full[2], "sample": sample},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS), help="BASELINE.json configuration (1..5)")
    ap.add_argument("--scene", default="", help="scene name under scenes/ (overrides --config)")
    ap.add_argument("--spp", type=int, default=-1, help="override SAMPLES of the scene")
    ap.add_argument("--width", type=int, default=-1)
    ap.add_argument("--height", type=int, default=-1)
    ap.add_argument("--batch-paths", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-peaks", action="store_true", help="skip the live roof measurement (tools/peaks)")
    ap.add_argument("--no-cli", action="store_true", help="skip the run.sh wall-time measurement")
    ap.add_argument("--ref-width", type=int, default=64)
    ap.add_argument("--ref-height", type=int, default=64)
    ap.add_argument("--ref-spp", type=int, default=8)
    ap.add_argument("--traversal", type=int, default=0)
    ap.add_argument("--frames-in-flight", type=int, default=2, choices=[1, 2],
                    help="device-resident timing: frames queued on alternating streams (every frame still complete in the timed region)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the radiance sums of the last device-resident timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return reference_arm(args, rank)

    import torch
    import torch.distributed as dist
    import raytracing_course_b200 as rtc

    if not torch.cuda.is_available() or rtc.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    cfg = resolve_config(args)
    path = scene_file(cfg["scene"])
    peaks = None if (args.no_peaks or rank != 0) else live_peaks(local_rank)
    t0 = time.perf_counter()
    scene = rtc.Scene(path=path, device=local_rank)
    load_s = time.perf_counter() - t0
    scene.override(cfg.get("width", -1), cfg.get("height", -1), cfg.get("spp", -1), -1)
    scene.set_traversal(args.traversal)
    if args.batch_paths:
        scene.set_batch_paths(args.batch_paths)
    W, H, spp, depth = scene.width, scene.height, scene.samples, scene.ray_depth
    lo, hi = rtc.shard_samples(spp, rank, world)   # spp sharding: rank r renders samples [lo, hi)
    npix = W * H
    nflight = args.frames_in_flight
    accums = [torch.zeros(npix * 3, dtype=torch.float32, device=dev) for _ in range(2)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def render_step(step, pipelined):
        """device-resident step: zero, render this rank's samples, reduce onto rank 0"""
        slot = step % nflight if pipelined else 0
        accum = accums[slot]
        if not pipelined:
            accum.zero_()
            scene.render_accumulate(accum.data_ptr(), seed=1000 + step, sample_begin=lo, sample_count=hi - lo)
            if world > 1:
                dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)
            return
        st = streams[slot]
        with torch.cuda.stream(st):
            accum.zero_()
            scene.render_accumulate(accum.data_ptr(), seed=1000 + step, sample_begin=lo, sample_count=hi - lo,
                                    stream=st.cuda_stream)
            if world > 1:
                dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)

    def timed(nsteps, first_step, pipelined):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        a.record()
        for st in streams:
            st.wait_stream(cur)
        for i in range(nsteps):
            render_step(first_step + i, pipelined)
        for st in streams:
            cur.wait_stream(st)
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def timed_e2e(nsteps, first_step):
        """host buffers in, host buffer out, frames queued two deep through rtc_frame_begin / rtc_frame_end; for
        N > 1 every rank uploads its scene and renders its samples, rank 0 reduces, resolves and reads back"""
        barrier()
        t0 = time.perf_counter()
        h2d = 0
        if world == 1:
            pending = []
            for i in range(nsteps):
                h2d = scene.frame_begin(seed=2000 + first_step + i, slot=i & 1)
                pending.append(i & 1)
                if len(pending) == 2:
                    scene.frame_end(pending.pop(0))
            while pending:
                scene.frame_end(pending.pop(0))
        else:
            cur = torch.cuda.current_stream()
            for st in streams:
                st.wait_stream(cur)
            for i in range(nsteps):
                accum, st = accums[i & 1], streams[i & 1]   # two frames in flight on alternating streams, as above
                h2d = scene.upload_async()
                with torch.cuda.stream(st):
                    accum.zero_()
                    scene.render_accumulate(accum.data_ptr(), seed=2000 + first_step + i, sample_begin=lo, sample_count=hi - lo,
                                            stream=st.cuda_stream)
                    dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)
                    if rank == 0:
                        scene.resolve_to_host(accum.data_ptr(), spp, stream=st.cuda_stream)
            for st in streams:
                cur.wait_stream(st)
            if rank == 0:
                scene.host_image_wait()
        barrier()
        ms = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), h2d

    # ---- warm-up (also sizes the wavefront buffers), then an untimed instrumented pass
    pipelined = nflight > 1
    for i in range(max(args.warmup, 3)):
        render_step(i, pipelined)
    barrier()
    scene.reset_counters()
    scene.set_profiling(kernel_events=False, count_visits=True)
    render_step(0, False)
    barrier()
    stats = scene.counters()
    lanes = scene.traverse_lanes()

    # ---- timed region: device-resident (no per-kernel events: they cost ~1 % of a step)
    scene.set_profiling(False, False)
    scene.reset_counters()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total = timed(args.steps, 100, pipelined)
    clocks = sampler.result()
    cnt = scene.counters()
    if args.dump_outputs and rank == 0:   # rank 0 holds the reduced sums; the passes below reuse the buffers
        last = 100 + args.steps - 1
        dump_outputs(args.dump_outputs, accums[last % nflight if pipelined else 0], W, H)
    # ---- the same steps again with CUDA events around every kernel (roofline durations)
    scene.set_profiling(kernel_events=True, count_visits=False)
    render_step(0, False)   # the single-stream pass may need larger wavefront buffers: allocate them untimed
    scene.profile()
    ms_profiled = timed(args.steps, 100, False)
    prof = scene.profile()
    scene.set_profiling(False, False)

    # ---- timed region: end to end through host buffers
    timed_e2e(2, 0)
    e2e_ms, h2d_bytes = timed_e2e(args.steps, 200)

    paths_rank = npix * (hi - lo) * args.steps
    t_paths = torch.tensor([float(paths_rank), float(cnt["rays"]), float(cnt["launches"]), float(h2d_bytes)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_paths, op=dist.ReduceOp.SUM)
    total_paths, total_rays, total_launches, h2d_bytes = [float(x) for x in t_paths.tolist()]   # whole job: every rank uploads its scene
    ms_per_step = ms_total / args.steps
    value = total_paths / (ms_total * 1e-3) / 1e6
    mrays = total_rays / (ms_total * 1e-3) / 1e6
    e2e_value = total_paths / (e2e_ms * 1e-3) / 1e6

    if rank == 0:
        rooflines, top = build_rooflines(scene, args, cnt, stats, lanes, prof, ms_profiled, peaks)
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = reference_arm(args, 0)
        cli_s = None
        if not args.no_cli and world == 1:
            cli_s = run_cli(path, cfg)
        line = {"metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": cfg["scene"], "baseline_config": args.config if not args.scene else None,
                           "width": W, "height": H, "spp": spp, "ray_depth": depth,
                           "paths_per_step": npix * spp, "triangles": scene.nbvh, "parallelism": "spp-shard x%d" % world,
                           "l2": "wavefront state (%.0f MB per bounce and batch) exceeds the 126 MB L2" % (min(npix * (hi - lo), 1 << 24) * 112 / 1e6),
                           "traversal": "index" if args.traversal == 0 else "reftree",
                           "frames_in_flight": nflight},
                "mrays_per_s": mrays, "rays_per_path": total_rays / max(total_paths, 1),
                "e2e": {"value": e2e_value, "unit": METRIC, "h2d_bytes_per_step": int(h2d_bytes),
                        "d2h_bytes_per_step": int(npix * 3), "ms_per_step": e2e_ms / args.steps,
                        "frames_in_flight": 2},
                "load_s": load_s, "cli_s": cli_s,
                "gpu_launches": int(total_launches), "fallback_rays": cnt["fallback_rays"],
                "clocks": clocks, "roofline": rooflines[top], "rooflines": rooflines, "peaks": peaks, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    scene.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_cli(path, cfg):
    """wall time of `run.sh <scene> <out.ppm>` (process start, parse, BVH builds, upload, render, PPM)"""
    env = dict(os.environ)
    for k, e in (("width", "RTC_WIDTH"), ("height", "RTC_HEIGHT"), ("spp", "RTC_SAMPLES")):
        if k in cfg:
            env[e] = str(cfg[k])
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        r = subprocess.run([os.path.join(ROOT, "run.sh"), path, os.path.join(tmp, "out.ppm")], env=env,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        dt = time.perf_counter() - t0
    return dt if r.returncode == 0 else None


def build_rooflines(scene, args, cnt, stats, lanes, prof, ms_profiled, peaks):
    """One roofline object per kernel class (DESIGN.md "Roofline"); returns (dict, key of the dominant kernel)."""
    hbm, hbm_src = hbm_peak()
    rays0 = max(cnt["rays"], 1)
    trav0 = max(cnt["traversed_rays"], 1)
    paths0 = max(cnt["paths"], 1)
    visits_per_ray = stats["index_node_visits"] / max(stats["traversed_rays"], 1)
    tests_per_ray = stats["prim_tests"] / max(stats["traversed_rays"], 1)
    node_bytes = scene.stats().get("index_node_bytes", 96)
    survive = max(rays0 - paths0, 0) / rays0          # rays that were written by k_shade (the others by k_generate)
    enter = trav0 / rays0
    ncu = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("workload") == scene_name_of(args):
            ncu = tj.get("kernels", {})
    except Exception:
        pass
    kname_trav = "k_traverse" if args.traversal == 0 else "k_extend_reftree"
    spec = {
        # key: (kernel, bound, algorithmic bytes per unit, units in the timed region, unit name)
        # a traverse-queue entry is the ray itself (32 B: origin | queue word, direction | plane distance), read once; 4 B of hit id out
        "traverse": (kname_trav, "l2", 32 + 4 + node_bytes * visits_per_ray + 48 * tests_per_ray, trav0, "ray entering the BVH"),
        # streamed state only: 52 B in, (48 + 4 + 32 * enter) B out per surviving ray; the winner's geometry and material
        # rows (80 B) are L2-resident and not counted
        "shade": ("k_shade", "hbm", 52 + (52 + 32 * enter) * survive, rays0, "ray"),
        "generate": ("k_generate", "hbm", 52 + 32 * enter, paths0, "camera path"),
    }
    out = {}
    for key, (kname, bound, bpu, units, uname) in spec.items():
        p = prof.get(key, {"ms": 0.0, "launches": 0})
        launches = max(p["launches"], 1)
        ms = p["ms"]
        per_launch_ms = ms / launches
        achieved = bpu * units / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        if bound == "l2":
            peak = peaks["l2_gather96_gbs"] if peaks else None
            src = (peaks["source"] + ": L2-resident random 96-byte gather over a 36 MB table") if peaks else "unavailable"
        else:
            peak, src = hbm, hbm_src
        n = ncu.get(kname, {})
        r = {"kernel": kname, "bound": bound, "achieved": achieved, "peak": peak, "unit": "GB/s",
             "frac": (achieved / peak) if peak else None, "peak_source": src,
             "traffic": n.get("dram_bytes_per_launch"), "bytes_per_unit": bpu, "unit_name": uname,
             "units_per_launch": units / launches, "avg_launch_ms": per_launch_ms, "launches": launches,
             "share_of_step": ms / ms_profiled if ms_profiled > 0 else None,
             "munits_per_s_in_kernel": units / (ms * 1e-3) / 1e6 if ms > 0 else None}
        # Per-launch figures of the committed ncu launch list of this same command (profiles/traffic.json); the launches of a
        # kernel are statistically alike from frame to frame, so "per launch" there and here mean the same work.
        if bound == "hbm" and n.get("dram_bytes_per_launch") and per_launch_ms > 0:
            # the same fraction on MEASURED DRAM traffic
            r["achieved_on_traffic"] = n["dram_bytes_per_launch"] / (per_launch_ms * 1e-3) / 1e9
            r["frac_on_traffic"] = r["achieved_on_traffic"] / peak if peak else None
        if n.get("warp_inst_per_launch") and peaks and per_launch_ms > 0:
            gw = n["warp_inst_per_launch"] / (per_launch_ms * 1e-3) / 1e9
            r["issue"] = {"warp_inst_per_unit": n["warp_inst_per_launch"] / max(units / launches, 1), "achieved_gwinst_s": gw,
                          "peak_gwinst_s": peaks["ffma_gwinst_s"], "frac": gw / peaks["ffma_gwinst_s"],
                          "lanes_per_32_ncu": n.get("lanes_per_inst"), "issue_active_pct_ncu": n.get("issue_active_pct")}
        if n.get("l1_wavefronts_pct"):
            r["l1_data_pipe_pct_ncu"] = n["l1_wavefronts_pct"]
        if key == "traverse":
            r.update({"index_node_visits_per_traversed_ray": visits_per_ray, "prim_tests_per_traversed_ray": tests_per_ray,
                      "traversed_fraction_of_rays": enter, "scheduler_lanes_of_32": lanes})
        out[key] = r
    kernel_ms = {k: v["ms"] / args.steps for k, v in prof.items()}
    top = max(out, key=lambda k: prof.get(k, {"ms": 0})["ms"])
    for r in out.values():
        r["profiled_ms_per_step"] = ms_profiled / args.steps
        r["kernel_ms_per_step"] = kernel_ms
    return out, top


def scene_name_of(args):
    return args.scene if args.scene else CONFIGS[args.config]["scene"]


if __name__ == "__main__":
    sys.exit(main())
