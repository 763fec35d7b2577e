"""lens_bench.py -- what the thin lens costs on the 100k dragon.

512 x 512 at 128 spp, focused on the dragon (f = the forward distance of the centre pixel's primary hit).  One JSON line
per run:
  pinhole                 the scene without a lens: Render (camera rays from the per-pixel candidate lists)
  pinhole, views          RenderViews([the scene's camera]): the views path builds no lists, every camera ray takes
                          pre_step and k_traverse
  lens N px               Render with the lens (lens renders build no lists)
  lens N px, views        RenderViews([the scene's camera]) with the lens
for two apertures, given as the blur radius of the far background in pixels (3 and 30).  Per line:
  ms                      median of --repeats synchronous calls (each returns with the 8-bit image on the host), after
                          one warm-up call
  listed_share            camera rays resolved from lists / camera paths (the paths of bounce 1)
  list_lengths            share of pixels marked for the index traversal, and percentiles of the other lengths
  kernel_ms               k_generate ("generate") and k_pixel_candidates ("lists") per render, from profile() in a
                          separate profiled call
and the GPU's name and power limit, read in the same run.

  python tools/lens_bench.py [--out FILE] [--repeats 10]
"""
import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracing_course_b200 as rtc  # noqa: E402
from adaptive_bench import device_info, median_ms, scene_file  # noqa: E402

SCENE = "practice5_dragon_100k"
SIZE, SPP, SEED = 512, 128, 1
BLURS = [3, 30]
TRAVERSE = 0xFFFFFFFF


def focus(s):
    o, d = s.cam.GetToRay(np.array([[s.width / 2, s.height / 2]], np.float32))
    pid, t, _, _ = s.RayIntersection(o, d)
    assert pid[0] >= 0, "the centre ray misses the dragon"
    return float(t[0])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--repeats", type=int, default=10)
    args = ap.parse_args()
    if rtc.device_count() < 1:
        raise SystemExit("lens_bench.py needs a CUDA device")
    name, power = device_info()
    out = open(args.out, "w") if args.out else None

    def emit(line):
        line.update({"scene": SCENE, "width": SIZE, "height": SIZE, "spp": SPP, "gpu": name, "power_limit": power})
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n")
            out.flush()

    s = rtc.Scene(path=scene_file(SCENE), device=0)
    s.override(SIZE, SIZE, SPP)
    f = focus(s)
    tan_half = math.tan(float(s.camera()[12]) / 2)
    paths = SIZE * SIZE * SPP

    def run(case, r, views):
        s.set_lens(r, f)
        call = (lambda: s.RenderViews([s.camera()], seed=SEED)) if views else (lambda: s.Render(seed=SEED))
        ms, all_ms = median_ms(call, args.repeats)
        s.reset_counters()
        call()
        listed = s.camera_list_rays() / paths
        s.set_profiling(kernel_events=True)
        call()
        prof = s.profile()
        s.set_profiling(kernel_events=False)
        line = {"case": case, "aperture_radius": r, "focus_distance": f, "ms": round(ms, 3), "all_ms": [round(x, 3) for x in all_ms],
                "mpaths_per_s": round(paths / ms / 1e3, 1), "listed_share": round(listed, 4),
                "kernel_ms": {"generate": round(prof["generate"]["ms"], 3), "lists": round(prof["pre"]["ms"], 3),
                              "traverse": round(prof["traverse"]["ms"], 3), "shade": round(prof["shade"]["ms"], 3)}}
        if not views:
            lengths = s.camera_list_lengths().ravel()
            kept = lengths[lengths != TRAVERSE]
            line["list_lengths"] = {"traverse_share": round(float((lengths == TRAVERSE).mean()), 4),
                                    "p50": int(np.percentile(kept, 50)) if kept.size else None,
                                    "p90": int(np.percentile(kept, 90)) if kept.size else None,
                                    "max": int(kept.max()) if kept.size else None,
                                    "mean": round(float(kept.mean()), 2) if kept.size else None}
        emit(line)

    run("pinhole", 0.0, False)
    run("pinhole, views", 0.0, True)
    for blur in BLURS:
        r = blur * 2 * f * tan_half / SIZE
        run("lens %d px" % blur, r, False)
        run("lens %d px, views" % blur, r, True)
    s.close()


if __name__ == "__main__":
    main()
