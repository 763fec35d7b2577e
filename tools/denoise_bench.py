"""denoise_bench.py -- time and quality of the non-local-means denoiser (rtc_render_denoised) against the uniform render.

One JSON line per (scene, spp) and one "summary" line per scene:
  times        host clock around synchronous calls after one warm-up call each, the median of --repeats calls:
               rtc_render_u8 (uniform), rtc_render_denoised (uniform, every pixel at spp) at each strength, and the
               filter's own time = rtc_render_denoised(k) - rtc_render_denoised(0) (strength 0 skips the filter)
  quality      RMSE, in the squash space x / (1 + x) of tests/test_gpu_parity.py, of the per-pixel means against a render
               of ours at 4x the maximum sample count with another seed (tools/adaptive_bench.py's reference); and the
               relative change of the frame mean in squash space from the raw render to the denoised one (the filter
               should not change the frame's brightness)
  summary      per strength the equal-quality cost: the smallest spp whose denoised RMSE is at or below the uniform
               render's at the maximum spp, and the time of that call over the uniform render's at the maximum; and one
               row of adaptive sampling (tolerance 1/255, 16 samples first) plus the filter at the recommended strength
  device       name and power limit of the GPU, read in the same run

  python tools/denoise_bench.py [--out FILE] [--repeats 5]

With --devices 1,2,4,8 it measures rtc_render_denoised_multi at the recommended strength instead, one JSON line per
(scene, spp, device count); every time is the median of --repeats calls after one warm-up call:
  denoised_multi_ms    rtc_render_denoised_multi (image only: no mean, halves or spp copies)
  filter_multi_ms      the same minus the call at strength 0 (which skips the filter)
  route_ms             what a caller had to do without it: rtc_render_adaptive_multi with the halves and spp copied to the
                       host, then rtc_denoise, which copies them back up to one device and filters the whole frame there
  uniform_multi_ms     rtc_render_u8_multi at the same samples per pixel
  one_device_ms        rtc_render_denoised on device 0, and one_device_filter_ms its filter time (as filter_multi_ms)
  devices              the list passed; a count above the physical devices lists them round-robin (replicas of the scene
                       on one device, each on its own streams: such a run measures the cost of the split and the saved
                       host round trip, not scaling over GPUs)
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracing_course_b200 as rtc  # noqa: E402
from adaptive_bench import device_info, median_ms, rmse, scene_file, squash  # noqa: E402

# (scene, width, height, max samples); -1 keeps the scene file's value
SCENES = [("practice5_1", -1, -1, -1), ("practice5_dragon_100k", 512, 512, 128), ("practice5_dragon_100k_glass", 512, 512, 128)]
SPPS = [4, 8, 16, 32]
STRENGTHS = [0.25, 0.45, 0.7, 1.0]
SEED, REF_SEED = 1, 977
# (scene, width, height, samples per pixel) of the --devices run
MULTI_ROWS = [("practice5_dragon_100k_metal", 3840, 2160, 8), ("practice5_dragon_100k_metal", 3840, 2160, 32),
              ("practice5_dragon_100k", 512, 512, 8), ("practice5_1", 1024, 768, 4)]


def squash_mean_shift(est, raw):
    ok = np.isfinite(est).all(2) & np.isfinite(raw).all(2)
    return float(squash(est[ok]).mean() / squash(raw[ok]).mean() - 1.0)


def entry(name, argtypes):
    fn = getattr(C.CDLL(rtc.LIB_PATH), name)
    fn.restype = C.c_int
    fn.argtypes = argtypes
    return fn


def multi_main(args, emit):
    P, U32, F32, I = C.c_void_p, C.c_uint32, C.c_float, C.c_int
    denoised_multi = entry("rtc_render_denoised_multi", [P, P, I, U32, F32, U32, U32, F32, P, P, P, P, P])
    adaptive_multi = entry("rtc_render_adaptive_multi", [P, P, I, U32, F32, U32, U32, P, P, P, P])
    denoise = entry("rtc_denoise", [P, P, P, F32, P, P])
    denoised = entry("rtc_render_denoised", [P, U32, F32, U32, U32, F32, P, P, P])
    physical = rtc.device_count()
    counts = [int(v) for v in args.devices.split(",")]
    k = rtc.DENOISE_STRENGTH

    def ok(s, rc):
        if rc:
            raise rtc.RtcError(s.lib.rtc_last_error().decode())
    for scene, w, h, spp in MULTI_ROWS:
        s = rtc.Scene(path=scene_file(scene), device=0)
        s.override(w, h, spp)
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        img = np.zeros((h, w, 3), np.uint8)
        halves = np.zeros((h, w, 2, 3), np.float32)
        n = np.zeros((h, w), np.uint32)
        one_ms, _ = median_ms(lambda: ok(s, denoised(s.h, SEED, 0.0, spp, 0, k, ptr(img), None, None)), args.repeats)
        one_k0_ms, _ = median_ms(lambda: ok(s, denoised(s.h, SEED, 0.0, spp, 0, 0.0, ptr(img), None, None)), args.repeats)
        for ndev in counts:
            devices = [i % physical for i in range(ndev)]
            dv = np.asarray(devices, np.int32)

            def multi(strength):
                ok(s, denoised_multi(s.h, ptr(dv), ndev, SEED, 0.0, spp, 0, strength, ptr(img), None, None, None, None))

            def route():
                ok(s, adaptive_multi(s.h, ptr(dv), ndev, SEED, 0.0, spp, 0, None, ptr(halves), ptr(n), None))
                ok(s, denoise(s.h, ptr(halves), ptr(n), k, ptr(img), None))
            multi_ms, multi_all = median_ms(lambda: multi(k), args.repeats)
            k0_ms, _ = median_ms(lambda: multi(0.0), args.repeats)
            route_ms, _ = median_ms(route, args.repeats)
            uniform_ms, _ = median_ms(lambda: s.RenderMulti(devices, seed=SEED), args.repeats)
            emit({"kind": "multi", "scene": scene, "width": w, "height": h, "spp": spp, "strength": k, "ndev": ndev,
                  "devices": devices, "physical_devices": physical, "denoised_multi_ms": round(multi_ms, 3),
                  "denoised_multi_ms_all": [round(t, 3) for t in multi_all], "denoised_multi_k0_ms": round(k0_ms, 3),
                  "filter_multi_ms": round(multi_ms - k0_ms, 3), "route_ms": round(route_ms, 3),
                  "uniform_multi_ms": round(uniform_ms, 3), "one_device_ms": round(one_ms, 3),
                  "one_device_filter_ms": round(one_ms - one_k0_ms, 3),
                  "denoised_multi_over_route": round(multi_ms / route_ms, 4),
                  "denoised_multi_over_uniform_multi": round(multi_ms / uniform_ms, 4)})
        s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--devices", default="", help="device counts, e.g. 1,2,4,8: measure rtc_render_denoised_multi")
    args = ap.parse_args()
    if rtc.device_count() < 1:
        raise SystemExit("denoise_bench.py needs a CUDA device")
    name, power = device_info()
    # the denoised call without the mean output (its copy to the host is not part of the timed render)
    raw = C.CDLL(rtc.LIB_PATH).rtc_render_denoised
    raw.restype = C.c_int
    raw.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lines = []

    def emit(line):
        line.update(device=name, power_limit=power)
        print(json.dumps(line), flush=True)
        lines.append(line)

    scenes = [] if args.devices else SCENES   # --devices measures the multi-device call only
    for scene, w, h, smax in scenes:
        s = rtc.Scene(path=scene_file(scene), device=0)
        s.override(w, h, smax)
        smax = s.samples
        img = np.zeros((s.height, s.width, 3), np.uint8)
        ref = s.RenderSum(seed=REF_SEED, sample_count=4 * smax).astype(np.float64) / (4 * smax)
        rows = []
        for spp in sorted(set(SPPS + [smax])):
            if spp > smax:
                continue
            s.override(-1, -1, spp)

            def denoised(k, tolerance=0.0, min_samples=spp):
                rc = raw(s.h, SEED, tolerance, min_samples, 0, k, img.ctypes.data_as(C.c_void_p), None, None)
                if rc:
                    raise rtc.RtcError(s.lib.rtc_last_error().decode())
            uniform_ms, _ = median_ms(lambda: s.Render(seed=SEED), args.repeats)
            raw_mean = s.RenderSum(seed=SEED, sample_count=spp).astype(np.float64) / spp
            zero_ms, _ = median_ms(lambda: denoised(0.0), args.repeats)
            row = {"kind": "spp", "scene": scene, "width": s.width, "height": s.height, "spp": spp, "max_samples": smax,
                   "uniform_ms": round(uniform_ms, 3), "rmse_uniform": rmse(raw_mean, ref), "denoised_k0_ms": round(zero_ms, 3),
                   "strengths": {}}
            for k in STRENGTHS:
                ms, _ = median_ms(lambda: denoised(k), args.repeats)
                mean = s.RenderDenoised(k, seed=SEED)[1].astype(np.float64)
                row["strengths"][str(k)] = {"denoised_ms": round(ms, 3), "filter_ms": round(ms - zero_ms, 3), "rmse": rmse(mean, ref),
                                            "squash_mean_shift": squash_mean_shift(mean, raw_mean)}
            row["reference"] = "ours, %d spp, seed %d" % (4 * smax, REF_SEED)
            emit(row)
            rows.append(row)
        s.override(-1, -1, smax)
        full = [r for r in rows if r["spp"] == smax][0]
        summary = {"kind": "summary", "scene": scene, "width": s.width, "height": s.height, "max_samples": smax,
                   "rmse_uniform_max": full["rmse_uniform"], "uniform_max_ms": full["uniform_ms"], "equal_quality": {}}
        for k in STRENGTHS:
            hit = [r for r in rows if r["strengths"][str(k)]["rmse"] <= full["rmse_uniform"]]
            if hit:
                r = hit[0]
                summary["equal_quality"][str(k)] = {"spp": r["spp"], "denoised_ms": r["strengths"][str(k)]["denoised_ms"],
                                                    "time_over_uniform_max": round(r["strengths"][str(k)]["denoised_ms"] / full["uniform_ms"], 4)}
            else:
                summary["equal_quality"][str(k)] = None
        k = rtc.DENOISE_STRENGTH
        ad_ms, _ = median_ms(lambda: denoised(k, 1 / 255, 16), args.repeats)
        mean, st = s.RenderDenoised(k, tolerance=1 / 255, min_samples=16, seed=SEED)[1:]
        summary["adaptive_denoised"] = {"tolerance": 1 / 255, "min_samples": 16, "strength": k, "ms": round(ad_ms, 3),
                                        "time_over_uniform_max": round(ad_ms / full["uniform_ms"], 4), "paths": st["paths"],
                                        "paths_over_uniform": round(st["paths"] / (s.width * s.height * smax), 4),
                                        "rmse": rmse(mean.astype(np.float64), ref)}
        emit(summary)
        s.close()
    if args.devices:
        multi_main(args, emit)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
