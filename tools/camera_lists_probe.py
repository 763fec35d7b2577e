"""tools/camera_lists_probe.py -- where camera rays stand in the traversal, and how long the per-pixel candidate lists are.

On one GPU, one JSON line per measurement:
  * "depth": per BASELINE.json dragon configuration (2, 3, 4) at RAY_DEPTH 1 and at the scene's own depth, the per-kernel
    CUDA-event times per frame (generate / traverse / shade / other, one stream), the rays the traverse queue took and,
    where the build has them, the camera rays resolved from candidate lists;
  * "lists": per configuration the distribution of the candidate-list lengths over the pixels of the scene's camera
    (k_pixel_candidates), the pixels whose rays take the index traversal, and the time of building the lists.
Runs from any build of the project: a build without candidate lists reports the "depth" lines only.

  python tools/camera_lists_probe.py [--configs 2,3,4] [--frames 5] > profiles/<name>.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import raytracing_course_b200 as rtc  # noqa: E402

SCENES = {2: "practice5_dragon_10k", 3: "practice5_dragon_100k", 4: "practice5_dragon_100k_glass"}


def gpu_name():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def render(s, frames, seed0):
    import torch
    accum = torch.zeros(s.width * s.height * 3, dtype=torch.float32, device="cuda")
    for i in range(frames):
        accum.zero_()
        s.render_accumulate(accum.data_ptr(), seed=seed0 + i, sample_begin=0, sample_count=s.samples)
    torch.cuda.synchronize()


def depth_line(cfg, depth, frames, card):
    s = rtc.Scene(path=os.path.join(ROOT, "scenes", SCENES[cfg] + ".txt"), device=0)
    s.override(512, 512, 128, depth)
    render(s, 2, 1)   # warm-up, sizes the buffers
    s.set_profiling(kernel_events=True, count_visits=False)
    s.profile()
    s.reset_counters()
    render(s, frames, 100)
    prof = s.profile()
    cnt = s.counters()
    s.set_profiling(False, False)
    line = {"kind": "depth", "config": cfg, "scene": SCENES[cfg], "ray_depth": s.ray_depth, "frames": frames, "gpu": card,
            "ms_per_frame": {k: v["ms"] / frames for k, v in prof.items()},
            "paths_per_frame": cnt["paths"] / frames, "rays_per_frame": cnt["rays"] / frames,
            "traversed_rays_per_frame": cnt["traversed_rays"] / frames, "fallback_rays": cnt["fallback_rays"]}
    if hasattr(s, "camera_list_rays"):
        line["list_rays_per_frame"] = s.camera_list_rays() / frames
    return line


def lists_line(cfg, card):
    s = rtc.Scene(path=os.path.join(ROOT, "scenes", SCENES[cfg] + ".txt"), device=0)
    s.override(512, 512, 128, -1)
    s.camera_list_lengths()   # warm-up
    t0 = time.perf_counter()
    n = s.camera_list_lengths()
    call_ms = (time.perf_counter() - t0) * 1e3
    trav = n == 0xFFFFFFFF
    lens = n[~trav].astype(np.int64)
    hist = np.bincount(lens, minlength=25).tolist() if lens.size else []
    return {"kind": "lists", "config": cfg, "scene": SCENES[cfg], "width": s.width, "height": s.height, "gpu": card,
            "pixels": int(n.size), "traverse_pixels": int(trav.sum()),
            "mean_length": float(lens.mean()) if lens.size else None,
            "percentiles_50_90_99_max": [int(np.percentile(lens, q)) for q in (50, 90, 99, 100)] if lens.size else None,
            "zero_length_pixels": int((lens == 0).sum()), "histogram": hist,
            "call_ms_incl_copy": call_ms}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="2,3,4")
    ap.add_argument("--frames", type=int, default=5)
    args = ap.parse_args()
    rtc.load_library()
    card = gpu_name()
    for cfg in [int(c) for c in args.configs.split(",")]:
        for depth in (1, -1):
            print(json.dumps(depth_line(cfg, depth, args.frames, card)), flush=True)
        s = rtc.Scene(path=os.path.join(ROOT, "scenes", SCENES[cfg] + ".txt"), device=0)
        if hasattr(s, "camera_list_lengths"):
            print(json.dumps(lists_line(cfg, card)), flush=True)


if __name__ == "__main__":
    main()
