"""views_bench.py -- what rendering one loaded scene from many cameras costs, three ways, on the 100k dragon.

One JSON line per (frame size, number of views V) over an orbit of V cameras around the dragon, 16 spp:
  reload_ms       (a) what a caller without a camera override does: for each view, load the scene text with its CAMERA_*
                  lines edited (reader, reference BVH, index BVH, upload) and render it.  Timed on the first
                  min(V, --reload-views) views and scaled to V (`reload_views_timed` says how many were timed)
  set_camera_ms   (b) set_camera + Render for each view, one after another
  views_ms        (c) one RenderViews call over all V views
  *_per_view_ms   the same over V; speedup_c_over_b = set_camera_ms / views_ms
Every (b) and (c) time is the median of --repeats calls after one warm-up call; (a) is one pass (its first load is a
warm-up load of the same text, not timed).  The host clock brackets synchronous calls (each returns with the 8-bit
images on the host).

One "rebuild" line: set_camera with a camera beyond the extent the index BVH was built for (the host rebuild of the
index BVH, the new arena and its upload), on a freshly loaded scene for each of 100x, 1000x and 10000x the file's
camera distance; and set_camera of a camera inside the extent (no rebuild) for comparison.

Each line carries the GPU's name and power limit, read in the same run.

  python tools/views_bench.py [--out FILE] [--repeats 3] [--reload-views 8]
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import raytracing_course_b200 as rtc  # noqa: E402
from adaptive_bench import device_info, median_ms, scene_file  # noqa: E402

SCENE = "practice5_dragon_100k"
SIZES = [128, 512]
VIEWS = [1, 8, 64]
SPP = 16
SEED = 1


def orbit(cam, angle):
    """`cam` turned by `angle` about the vertical axis through the point |pos| ahead of it (the dragon's origin)."""
    cam = np.asarray(cam, np.float64)
    pos, fwd = cam[0:3], cam[9:12]
    pivot = pos + fwd / np.linalg.norm(fwd) * np.linalg.norm(pos)
    c, s = math.cos(angle), math.sin(angle)
    rot = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])
    return np.concatenate([pivot + rot @ (pos - pivot), rot @ cam[3:6], rot @ cam[6:9], rot @ fwd, cam[12:13]]).astype(np.float32)


def with_camera(text, cam, size):
    vals = {"CAMERA_POSITION": cam[0:3], "CAMERA_RIGHT": cam[3:6], "CAMERA_UP": cam[6:9], "CAMERA_FORWARD": cam[9:12],
            "CAMERA_FOV_X": cam[12:13]}
    out = []
    for line in text.splitlines():
        word = line.split()[0] if line.split() else ""
        if word in vals:
            line = word + " " + " ".join("%.9g" % float(v) for v in vals[word])
        elif word == "DIMENSIONS":
            line = "DIMENSIONS %d %d" % (size, size)
        elif word == "SAMPLES":
            line = "SAMPLES %d" % SPP
        out.append(line)
    return "\n".join(out) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--reload-views", type=int, default=8)
    args = ap.parse_args()
    if rtc.device_count() < 1:
        raise SystemExit("views_bench.py needs a CUDA device")
    name, power = device_info()
    out = open(args.out, "w") if args.out else None

    def emit(line):
        line.update({"gpu": name, "power_limit": power})
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n")
            out.flush()

    text = open(scene_file(SCENE)).read()
    for size in SIZES:
        s = rtc.Scene(path=scene_file(SCENE), device=0)
        s.override(size, size, SPP)
        base = s.camera()
        for nv in VIEWS:
            cams = np.stack([orbit(base, 2 * math.pi * v / nv) for v in range(nv)])
            # (a) reload the edited text for each view
            rtc.Scene(text=with_camera(text, cams[0], size), device=0).close()
            k = min(nv, args.reload_views)
            t0 = time.perf_counter()
            for v in range(k):
                r = rtc.Scene(text=with_camera(text, cams[v], size), device=0)
                r.Render(seed=SEED)
                r.close()
            reload_ms = (time.perf_counter() - t0) * 1e3 * nv / k

            # (b) set_camera + Render per view
            def per_view():
                for v in range(nv):
                    s.set_camera(cams[v])
                    s.Render(seed=SEED)
            b_ms, b_all = median_ms(per_view, args.repeats)
            # (c) one batched call
            c_ms, c_all = median_ms(lambda: s.RenderViews(cams, seed=SEED), args.repeats)
            emit({"case": "views", "scene": SCENE, "width": size, "height": size, "spp": SPP, "views": nv,
                  "reload_ms": round(reload_ms, 2), "reload_views_timed": k, "set_camera_ms": round(b_ms, 3),
                  "views_ms": round(c_ms, 3), "reload_per_view_ms": round(reload_ms / nv, 2),
                  "set_camera_per_view_ms": round(b_ms / nv, 3), "views_per_view_ms": round(c_ms / nv, 3),
                  "speedup_c_over_b": round(b_ms / c_ms, 3), "set_camera_all_ms": [round(x, 3) for x in b_all],
                  "views_all_ms": [round(x, 3) for x in c_all], "mpaths_per_s_views": round(nv * size * size * SPP / c_ms / 1e3, 1)})
        s.close()

    rebuild = {}
    for k in (100, 1000, 10000):
        s = rtc.Scene(path=scene_file(SCENE), device=0)
        s.override(128, 128, SPP)
        cam = s.camera().copy()
        s.Render(seed=SEED)
        inside = orbit(cam, 0.5)
        t0 = time.perf_counter()
        s.set_camera(inside)
        inside_ms = (time.perf_counter() - t0) * 1e3
        cam[0:3] *= k
        cam[12] = 2 * math.atan(math.tan(float(cam[12]) / 2) / k)
        t0 = time.perf_counter()
        s.set_camera(cam)
        rebuild[str(k)] = round((time.perf_counter() - t0) * 1e3, 2)
        rebuild["inside_extent_%d" % k] = round(inside_ms, 3)
        assert s.arena_check() == 0
        s.close()
    emit({"case": "rebuild", "scene": SCENE, "set_camera_far_ms": rebuild})


if __name__ == "__main__":
    main()
