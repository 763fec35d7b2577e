"""adaptive_bench.py -- time and quality of adaptive sampling (rtc_render_adaptive) against the uniform render.

One JSON line per (scene, tau):
  times        host clock around the (synchronous) adaptive call and around rtc_render_u8 at the same maximum sample
               count, after one warm-up call each; the median of --repeats calls
  paths        paths the adaptive render traced, passes, tiles and tiles that stopped below the maximum
  quality      RMSE, in the squash space x / (1 + x) of tests/test_gpu_parity.py, of the per-pixel means against a render
               of ours at 4x the maximum sample count with another seed: for the adaptive image, for the uniform render
               at the maximum, and for a uniform render that traces about as many paths as the adaptive one
  device       name and power limit of the GPU, read in the same run

  python tools/adaptive_bench.py [--out FILE] [--repeats 5]

With --devices 1,2,4,8 it measures rtc_render_adaptive_multi instead, one JSON line per (scene, tau, device count):
  times        host clock around rtc_render_adaptive_multi (without the halves and spp outputs) and around
               rtc_render_u8_multi on the same device list; the first call of each is the warm-up (the adaptive one
               also gives the stats and the spp map), then the median of --repeats calls (one at 4K)
  paths        passes (the most of any device), paths, tiles stopped; path_spread = the largest share of the paths any
               device traced over the mean share, from the spp map and the ownership of tile t by device t % n
  quality      as above; the reference is RenderMulti over every physical device at 4x the maximum sample count
  devices      the list passed; a count above the physical devices lists them round-robin (replicas of the scene on
               one device run concurrently on its own streams, so such a run measures the overhead of the split, not
               its scaling)
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_course_b200 as rtc  # noqa: E402

# (scene, width, height, max samples); -1 keeps the scene file's value
SCENES = [("practice5_1", -1, -1, -1), ("practice5_dragon_100k", 512, 512, 128), ("practice5_dragon_100k_glass", -1, -1, -1)]
TAUS = [0.0, 1 / 255, 4 / 255]
SEED, REF_SEED, UNIFORM_SEED = 1, 977, 2


def device_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        power = r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def squash(x):
    return x / (1.0 + x)


def rmse(est, ref):
    ok = np.isfinite(est) & np.isfinite(ref)
    return float(np.sqrt(np.mean((squash(est[ok]) - squash(ref[ok])) ** 2)))


# (scene, width, height, max samples, taus, repeats or None for --repeats) of the --devices run
MULTI_SCENES = [("practice5_1", -1, -1, -1, TAUS, None), ("practice5_dragon_100k", 512, 512, 128, TAUS, None),
                ("practice5_dragon_100k_metal", 3840, 2160, 1024, [1 / 255], 1)]


def median_ms(fn, repeats, warm=True):
    if warm:
        fn()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), ts


def scene_file(scene):
    path = os.path.join(ROOT, "scenes", scene + ".txt")
    if not os.path.exists(path):
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_scenes.py")])
    return path


def path_spread(spp, ndev):
    """largest share of the paths any device traced over the mean share; tile t (row-major 8x8) is device t % ndev's"""
    h, w = spp.shape
    tiles_x = -(-w // 8)
    ys, xs = np.mgrid[0:h, 0:w]
    owner = ((ys // 8) * tiles_x + xs // 8) % ndev
    per_dev = np.bincount(owner.ravel(), weights=spp.astype(np.float64).ravel(), minlength=ndev)
    return float(per_dev.max() / per_dev.mean()), [int(v) for v in per_dev]


def multi_main(args, name, power):
    raw = C.CDLL(rtc.LIB_PATH).rtc_render_adaptive_multi
    raw.restype = C.c_int
    raw.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                    C.c_void_p, C.c_void_p]
    physical = rtc.device_count()
    counts = [int(v) for v in args.devices.split(",")]
    lines = []
    for scene, w, h, spp, taus, repeats in MULTI_SCENES:
        repeats = repeats or args.repeats
        s = rtc.Scene(path=scene_file(scene), device=0)
        s.override(w, h, spp)
        smax, npix = s.samples, s.width * s.height
        img = np.zeros((s.height, s.width, 3), np.uint8)
        s.override(-1, -1, 4 * smax)
        ref = s.RenderMulti(list(range(physical)), seed=REF_SEED, want_sum=True)[1].astype(np.float64) / (4 * smax)
        s.override(-1, -1, smax)
        rmse_full = rmse(s.RenderSum(seed=SEED, sample_count=smax).astype(np.float64) / smax, ref)
        for ndev in counts:
            devices = [i % physical for i in range(ndev)]
            dv = np.asarray(devices, np.int32)
            uniform_ms, uniform_all = median_ms(lambda: s.RenderMulti(devices, seed=SEED), repeats)
            for tau in taus:
                _, halves, n, st = s.RenderAdaptiveMulti(devices, tau, min_samples=args.min_samples, seed=SEED)   # warm-up

                def call():
                    rc = raw(s.h, dv.ctypes.data_as(C.c_void_p), ndev, SEED, tau, args.min_samples, 0,
                             img.ctypes.data_as(C.c_void_p), None, None, None)
                    if rc:
                        raise rtc.RtcError(s.lib.rtc_last_error().decode())
                adaptive_ms, adaptive_all = median_ms(call, repeats, warm=False)
                est = halves.sum(2).astype(np.float64) / n[:, :, None]
                eq_spp = max(1, int(round(st["paths"] / npix)))
                eq = s.RenderSum(seed=UNIFORM_SEED, sample_count=eq_spp).astype(np.float64) / eq_spp
                spread, per_dev = path_spread(n, ndev)
                line = {
                    "scene": scene, "width": s.width, "height": s.height, "max_samples": smax, "min_samples": args.min_samples,
                    "tau": tau, "tau_in_8bit_levels": tau * 255, "ndev": ndev, "devices": devices, "physical_devices": physical,
                    "adaptive_multi_ms": round(adaptive_ms, 3), "uniform_multi_ms": round(uniform_ms, 3),
                    "adaptive_over_uniform_time": round(adaptive_ms / uniform_ms, 4),
                    "adaptive_multi_ms_all": [round(t, 3) for t in adaptive_all],
                    "uniform_multi_ms_all": [round(t, 3) for t in uniform_all],
                    "passes": st["passes"], "paths": st["paths"], "uniform_paths": npix * smax,
                    "paths_over_uniform": round(st["paths"] / (npix * smax), 4),
                    "tiles": st["tiles"], "tiles_stopped": st["tiles_stopped"],
                    "path_spread": round(spread, 4), "paths_per_device": per_dev,
                    "spp_histogram": {str(int(k)): int(v) for k, v in zip(*np.unique(n, return_counts=True))},
                    "rmse_adaptive": rmse(est, ref), "rmse_uniform_max": rmse_full,
                    "equal_cost_spp": eq_spp, "rmse_uniform_equal_cost": rmse(eq, ref),
                    "reference": "ours, %d spp, seed %d" % (4 * smax, REF_SEED),
                    "device": name, "power_limit": power,
                }
                print(json.dumps(line), flush=True)
                lines.append(line)
        s.close()
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--min-samples", type=int, default=16)
    ap.add_argument("--devices", default="", help="device counts, e.g. 1,2,4,8: measure rtc_render_adaptive_multi")
    args = ap.parse_args()
    if rtc.device_count() < 1:
        raise SystemExit("adaptive_bench.py needs a CUDA device")
    name, power = device_info()
    lines = multi_main(args, name, power) if args.devices else single_main(args, name, power)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


def single_main(args, name, power):
    # the adaptive call without the optional outputs (the halves and spp copies are not part of the timed render)
    raw = C.CDLL(rtc.LIB_PATH).rtc_render_adaptive
    raw.restype = C.c_int
    raw.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lines = []
    for scene, w, h, spp in SCENES:
        s = rtc.Scene(path=scene_file(scene), device=0)
        s.override(w, h, spp)
        smax, npix = s.samples, s.width * s.height
        img = np.zeros((s.height, s.width, 3), np.uint8)
        uniform_ms, uniform_all = median_ms(lambda: s.Render(seed=SEED), args.repeats)
        ref = s.RenderSum(seed=REF_SEED, sample_count=4 * smax).astype(np.float64) / (4 * smax)
        full = s.RenderSum(seed=SEED, sample_count=smax).astype(np.float64) / smax
        rmse_full = rmse(full, ref)
        for tau in TAUS:
            def call():
                rc = raw(s.h, SEED, tau, args.min_samples, 0, img.ctypes.data_as(C.c_void_p), None, None, None)
                if rc:
                    raise rtc.RtcError(s.lib.rtc_last_error().decode())
            adaptive_ms, adaptive_all = median_ms(call, args.repeats)
            _, halves, n, st = s.RenderAdaptive(tau, min_samples=args.min_samples, seed=SEED)
            est = halves.sum(2).astype(np.float64) / n[:, :, None]
            eq_spp = max(1, int(round(st["paths"] / npix)))
            eq = s.RenderSum(seed=UNIFORM_SEED, sample_count=eq_spp).astype(np.float64) / eq_spp
            line = {
                "scene": scene, "width": s.width, "height": s.height, "max_samples": smax, "min_samples": args.min_samples,
                "tau": tau, "tau_in_8bit_levels": tau * 255,
                "adaptive_ms": round(adaptive_ms, 3), "uniform_ms": round(uniform_ms, 3),
                "adaptive_over_uniform_time": round(adaptive_ms / uniform_ms, 4),
                "adaptive_ms_all": [round(t, 3) for t in adaptive_all], "uniform_ms_all": [round(t, 3) for t in uniform_all],
                "passes": st["passes"], "paths": st["paths"], "uniform_paths": npix * smax,
                "paths_over_uniform": round(st["paths"] / (npix * smax), 4),
                "tiles": st["tiles"], "tiles_stopped": st["tiles_stopped"],
                "spp_histogram": {str(int(k)): int(v) for k, v in zip(*np.unique(n, return_counts=True))},
                "rmse_adaptive": rmse(est, ref), "rmse_uniform_max": rmse_full,
                "equal_cost_spp": eq_spp, "rmse_uniform_equal_cost": rmse(eq, ref),
                "reference": "ours, %d spp, seed %d" % (4 * smax, REF_SEED),
                "device": name, "power_limit": power,
            }
            print(json.dumps(line), flush=True)
            lines.append(line)
        s.close()
    return lines


if __name__ == "__main__":
    main()
