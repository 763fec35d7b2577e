"""Scene lifetime and the double scene arena, through the C-ABI (-m gpu).

rtc_scene_upload_async fills the arena that is not being read, on a copy stream of its own, and switches the scene to
it at once: every entry point whose kernels read the scene has to wait for that upload, and the next upload into an
arena has to wait for the kernels that read it.  A scene owns its CUDA resources and frees all of them when it is
closed, replicas made by RenderMulti included."""
import os
import subprocess

import numpy as np
import pytest

from conftest import scene_path

pytestmark = pytest.mark.gpu


def probe_inputs(s):
    """Seeded inputs of the four probes: primary rays of a pixel grid, the primitives a few of them hit, and the hit
    points, normals and directions of mix_distrib"""
    rng = np.random.default_rng(11)
    ys, xs = np.mgrid[0:s.height:8, 0:s.width:8]
    xy = np.stack([xs.ravel() + 0.5, ys.ravel() + 0.5], 1).astype(np.float32)
    o, d = s.cam.GetToRay(xy)
    pid, t, nrm, _ = s.RayIntersection(o, d)
    hit = pid >= 0
    assert hit.sum() > 100
    prims = [int(p) for p in rng.choice(np.unique(pid[hit]), 4, replace=False)]
    x = (o[hit] + t[hit, None] * d[hit]).astype(np.float32)
    dirs = rng.normal(size=x.shape).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    return xy, o, d, prims, x, nrm[hit].copy(), dirs


def probe_calls(s, xy, o, d, prims, x, nrm, dirs):
    """One callable per probe, each returning the bytes of its results"""
    def flat(*arrays):
        return b"".join(np.ascontiguousarray(a).tobytes() for a in arrays)
    calls = [lambda: flat(*s.cam.GetToRay(xy))]
    calls += [lambda p=p: flat(*s.PrimitiveIntersect(p, o, d)) for p in prims]
    calls.append(lambda: flat(s.mix_distrib.Pdf(x, nrm, dirs)))
    calls.append(lambda: flat(s.mix_distrib.Sample(x, nrm, seed=7, sample=3, bounce=2)))
    return calls


def test_probes_after_async_upload(rtc):
    """A probe issued right after rtc_scene_upload_async reads the scene only once the upload has landed: its results
    are bit for bit the ones of the resident scene, and the arena is intact afterwards."""
    s = rtc.Scene(path=scene_path("practice5_dragon_100k"), device=0)
    calls = probe_calls(s, *probe_inputs(s))
    want = [call() for call in calls]
    for _ in range(2):   # into the second arena (allocated and zeroed on the way), then back into the first
        for i, call in enumerate(calls):
            s.upload_async()
            assert call() == want[i], "probe %d differs after an asynchronous upload" % i
    assert s.arena_check() == 0
    s.close()


def device_mib():
    """This process's device memory in MiB as nvidia-smi lists it, or None when it does not list this process"""
    try:
        r = subprocess.run(["nvidia-smi", "--query-compute-apps=pid,used_memory", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
    except (OSError, subprocess.TimeoutExpired):
        return None
    for line in r.stdout.splitlines():
        fields = [f.strip() for f in line.split(",")]
        if len(fields) == 2 and fields[0] == str(os.getpid()) and fields[1].isdigit():
            return int(fields[1])
    return None


def exercise_and_free(rtc, torch):
    """Create a scene, run every path that acquires device resources, free it"""
    s = rtc.Scene(path=scene_path("practice5_dragon_100k"), device=0)
    s.override(96, 64, 4)
    stream = torch.cuda.current_stream().cuda_stream
    s.Render(seed=1)
    s.RenderAdaptive(0.01, min_samples=2, max_samples=4, seed=2)
    img = [np.zeros((s.height, s.width, 3), np.uint8) for _ in range(2)]
    s.frame_begin(seed=3, slot=0)
    s.frame_begin(seed=4, slot=1)
    s.frame_end(0, img[0])
    s.frame_end(1, img[1])
    accum = torch.zeros(s.height * s.width * 3, dtype=torch.float32, device="cuda")
    s.render_accumulate(accum.data_ptr(), 5, 0, 4, stream=stream)
    s.resolve_to_host(accum.data_ptr(), 4, stream=stream)
    s.host_image_wait(img[0])
    n = 4096
    rays = torch.randn((2, n, 3), dtype=torch.float32, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    out = [torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.float32, device="cuda"),
           torch.empty((n, 3), dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda")]
    s.intersect_dev(n, rays[0].data_ptr(), rays[1].data_ptr(), *[t.data_ptr() for t in out], stream=stream)
    torch.cuda.synchronize()
    s.RenderMulti([0, 0], seed=6)   # the second use of device 0 is a replica of the scene
    s.close()
    torch.cuda.synchronize()


def test_create_exercise_free_leaves_nothing_behind(rtc):
    import torch
    exercise_and_free(rtc, torch)   # warm-up: CUDA context, modules, torch's cached blocks
    first = device_mib()
    if first is None:
        pytest.skip("nvidia-smi does not list this process (pid %d), as in some containers" % os.getpid())
    for _ in range(3):
        exercise_and_free(rtc, torch)
    last = device_mib()
    assert last is not None and abs(last - first) <= 2, (first, last)
