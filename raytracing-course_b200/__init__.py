"""raytracing-course_b200 -- B200-native hot path of FeggieBoss/raytracing-course hw5.

The product is the C-ABI library ``librtc_b200.so`` (include/rtc_b200.h) and the
``raytracing_hw5`` command line next to it; both are built by ``csrc/Makefile``.  This module
is the thin ctypes binding used by tests/, bench.py and __graft_entry__.py.  Method names
mirror the reference's C++ interface (Scene::Load / InitScene / Render / RayIntersection,
Camera::GetToRay, Distribution::Pdf / Sample, AcesTonemap / GammaCorrected / toUInts) so that
the parity tests read like the reference's own call sites.

There is no CPU fallback: if the CUDA library is missing, importing works but every use raises
``RtcError`` (and ``load_library`` raises ``OSError``).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librtc_b200.so")
CLI_PATH = os.path.join(HERE, "raytracing_hw5")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "rtc_b200.h")

TRAVERSAL_INDEX = 0
TRAVERSAL_REFTREE = 1
# recommended strength of the denoiser (Scene.Denoise, Scene.RenderDenoised; DESIGN.md "Denoising")
DENOISE_STRENGTH = 0.45

_f32 = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32 = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u32 = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_u64 = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
_u8 = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")

_SIGNATURES = {
    "rtc_last_error": (C.c_char_p, []),
    "rtc_version": (C.c_int, []),
    "rtc_device_count": (C.c_int, []),
    "rtc_scene_load": (C.c_void_p, [C.c_char_p, C.c_int]),
    "rtc_scene_parse": (C.c_void_p, [C.c_char_p, C.c_long, C.c_int]),
    "rtc_scene_load_dialect": (C.c_void_p, [C.c_char_p, C.c_int, C.c_int]),
    "rtc_scene_parse_dialect": (C.c_void_p, [C.c_char_p, C.c_long, C.c_int, C.c_int]),
    "rtc_scene_dialect": (C.c_int, [C.c_void_p]),
    "rtc_scene_free": (None, [C.c_void_p]),
    "rtc_scene_upload": (C.c_int, [C.c_void_p, _u64]),
    "rtc_scene_info": (C.c_int, [C.c_void_p, _u32]),
    "rtc_scene_stats": (C.c_int, [C.c_void_p, _u64]),
    "rtc_scene_override": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "rtc_scene_prim_order": (C.c_int, [C.c_void_p, _i32]),
    "rtc_scene_prims": (C.c_int, [C.c_void_p, _i32, _f32]),
    "rtc_scene_nodes": (C.c_int, [C.c_void_p, _f32, _u32]),
    "rtc_scene_root": (C.c_uint32, [C.c_void_p]),
    "rtc_set_traversal": (None, [C.c_void_p, C.c_int]),
    "rtc_intersect": (C.c_int, [C.c_void_p, C.c_long, _f32, _f32, _i32, _f32, _f32, _i32, C.c_int]),
    "rtc_primitive_intersect": (C.c_int, [C.c_void_p, C.c_int, C.c_long, _f32, _f32, _i32, _f32, _f32, _i32]),
    "rtc_camera_rays": (C.c_int, [C.c_void_p, C.c_long, _f32, _f32, _f32]),
    "rtc_mix_pdf": (C.c_int, [C.c_void_p, C.c_long, _f32, _f32, _f32, _f32]),
    "rtc_mix_sample": (C.c_int, [C.c_void_p, C.c_long, _f32, _f32, C.c_uint32, C.c_uint32, C.c_uint32, _f32]),
    "rtc_tonemap_u8": (C.c_int, [C.c_void_p, C.c_long, _f32, _u8]),
    "rtc_render_accumulate": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "rtc_render_counters": (C.c_int, [C.c_void_p, C.c_void_p, _u64]),
    "rtc_render_reset_counters": (C.c_int, [C.c_void_p]),
    "rtc_traverse_lanes": (C.c_int, [C.c_void_p, C.c_void_p, _u64]),
    "rtc_scene_arena_check": (C.c_int, [C.c_void_p, _u64]),
    "rtc_intersect_dev": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_int, C.c_void_p]),
    "rtc_render_u8_multi": (C.c_int, [C.c_void_p, _i32, C.c_int, C.c_uint32, _u8, C.c_void_p]),
    "rtc_render_ppm_multi": (C.c_int, [C.c_void_p, _i32, C.c_int, C.c_uint32, C.c_char_p]),
    "rtc_scene_upload_async": (C.c_int, [C.c_void_p, _u64]),
    "rtc_frame_begin": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, _u64]),
    "rtc_frame_end": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "rtc_resolve_to_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "rtc_host_image_wait": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rtc_render_resolve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "rtc_render_u8": (C.c_int, [C.c_void_p, C.c_uint32, _u8]),
    "rtc_render_sum": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, _f32]),
    "rtc_render_ppm": (C.c_int, [C.c_void_p, C.c_uint32, C.c_char_p]),
    "rtc_render_adaptive": (C.c_int, [C.c_void_p, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, _u8, _f32, _u32, _u64]),
    "rtc_render_adaptive_multi": (C.c_int, [C.c_void_p, _i32, C.c_int, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, _u8, _f32,
                                            _u32, _u64]),
    "rtc_denoise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, _u8, C.c_void_p]),
    "rtc_render_denoised": (C.c_int, [C.c_void_p, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_float, _u8, C.c_void_p, _u64]),
    "rtc_render_denoised_multi": (C.c_int, [C.c_void_p, _i32, C.c_int, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_float, _u8,
                                            C.c_void_p, C.c_void_p, C.c_void_p, _u64]),
    "rtc_set_batch_paths": (C.c_int, [C.c_void_p, C.c_uint64]),
    "rtc_set_profiling": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "rtc_render_profile": (C.c_int, [C.c_void_p, C.c_void_p, np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS"), _u64, C.c_int]),
    "rtc_philox4x32_10": (None, [_u32, _u32, _u32]),
}


class RtcError(RuntimeError):
    pass


_lib = None


def load_library(path=None):
    """dlopen librtc_b200.so and declare every entry point of include/rtc_b200.h."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise OSError("CUDA library %s is missing: build it with `make -C %s` (no CPU fallback exists)"
                      % (p, os.path.join(HERE, "csrc")))
    lib = C.CDLL(p)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def _check(lib, rc):
    if rc != 0:
        raise RtcError("rtc error %d: %s" % (rc, lib.rtc_last_error().decode(errors="replace")))


def device_count():
    return load_library().rtc_device_count()


def _c3(a):
    a = np.ascontiguousarray(a, np.float32)
    if a.ndim != 2 or a.shape[1] != 3:
        raise ValueError("expected an (n, 3) float array")
    return a


class Camera:
    """Camera (include/scene.h:46-56) view of a Scene."""

    def __init__(self, scene):
        self._s = scene

    @property
    def width(self):
        return self._s.width

    @property
    def height(self):
        return self._s.height

    def GetToRay(self, xy):
        """Camera::GetToRay for an (n, 2) array of (x, y) -> origins (n,3), directions (n,3)."""
        xy = np.ascontiguousarray(xy, np.float32)
        n = xy.shape[0]
        o = np.zeros((n, 3), np.float32)
        d = np.zeros((n, 3), np.float32)
        _check(self._s.lib, self._s.lib.rtc_camera_rays(self._s.h, n, xy, o, d))
        return o, d


class Distribution:
    """Scene::mix_distrib (include/distributions.h:28-96)."""

    def __init__(self, scene):
        self._s = scene

    def Pdf(self, x, n, d):
        x, n, d = _c3(x), _c3(n), _c3(d)
        out = np.zeros(x.shape[0], np.float32)
        _check(self._s.lib, self._s.lib.rtc_mix_pdf(self._s.h, x.shape[0], x, n, d, out))
        return out

    def Sample(self, x, n, seed=0, sample=0, bounce=1):
        x, n = _c3(x), _c3(n)
        out = np.zeros(x.shape, np.float32)
        _check(self._s.lib, self._s.lib.rtc_mix_sample(self._s.h, x.shape[0], x, n, seed, sample, bounce, out))
        return out


class Scene:
    """Scene (include/scene.h:58-90): Load + InitScene happen in the constructor."""

    def __init__(self, path=None, text=None, device=0, dialect=5):
        """dialect 1..5: the homework snapshot whose scene vocabulary and Scene::RayTrace apply (5 = hw5)."""
        self.lib = load_library()
        self.dialect = dialect
        if path is not None:
            self.h = self.lib.rtc_scene_load_dialect(os.fsencode(path), device, dialect)
        elif text is not None:
            raw = text.encode() if isinstance(text, str) else bytes(text)
            self.h = self.lib.rtc_scene_parse_dialect(raw, len(raw), device, dialect)
        else:
            raise ValueError("path or text required")
        if not self.h:
            raise RtcError(self.lib.rtc_last_error().decode(errors="replace"))
        self.device = device
        self.cam = Camera(self)
        self.mix_distrib = Distribution(self)
        self._refresh()

    @classmethod
    def Load(cls, path, device=0, dialect=5):
        return cls(path=path, device=device, dialect=dialect)

    def _refresh(self):
        info = np.zeros(8, np.uint32)
        _check(self.lib, self.lib.rtc_scene_info(self.h, info))
        (self.width, self.height, self.ray_depth, self.samples,
         self.nprims, self.nbvh, self.nnodes, self.nlights) = [int(v) for v in info]

    def close(self):
        if getattr(self, "h", None):
            self.lib.rtc_scene_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- introspection ------------------------------------------------------------------
    def stats(self):
        out = np.zeros(8, np.uint64)
        _check(self.lib, self.lib.rtc_scene_stats(self.h, out))
        keys = ["index_nodes", "index_depth", "ref_depth", "units", "device_bytes", "lca_levels", "index_node_bytes", "features"]
        return dict(zip(keys, [int(v) for v in out[:8]]))

    def override(self, width=-1, height=-1, samples=-1, ray_depth=-1):
        _check(self.lib, self.lib.rtc_scene_override(self.h, width, height, samples, ray_depth))
        self._refresh()

    def prim_order(self):
        out = np.zeros(self.nprims, np.int32)
        _check(self.lib, self.lib.rtc_scene_prim_order(self.h, out))
        return out

    def prims(self):
        tm = np.zeros((self.nprims, 2), np.int32)
        d = np.zeros((self.nprims, 26), np.float32)
        _check(self.lib, self.lib.rtc_scene_prims(self.h, tm, d))
        return tm, d

    def nodes(self):
        aabb = np.zeros((self.nnodes, 6), np.float32)
        links = np.zeros((self.nnodes, 4), np.uint32)
        if self.nnodes:
            _check(self.lib, self.lib.rtc_scene_nodes(self.h, aabb, links))
        return aabb, links, int(self.lib.rtc_scene_root(self.h))

    def upload(self):
        out = np.zeros(1, np.uint64)
        _check(self.lib, self.lib.rtc_scene_upload(self.h, out))
        return int(out[0])

    def set_traversal(self, mode):
        self.lib.rtc_set_traversal(self.h, mode)

    def set_batch_paths(self, paths):
        _check(self.lib, self.lib.rtc_set_batch_paths(self.h, int(paths)))

    # ---- hot path -------------------------------------------------------------------------
    def RayIntersection(self, o, d, mode=TRAVERSAL_INDEX):
        """Scene::RayIntersection for n rays -> (id, t, normal, interior); id = -1 on a miss."""
        o, d = _c3(o), _c3(d)
        n = o.shape[0]
        pid = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        nrm = np.zeros((n, 3), np.float32)
        inter = np.zeros(n, np.int32)
        _check(self.lib, self.lib.rtc_intersect(self.h, n, o, d, pid, t, nrm, inter, mode))
        return pid, t, nrm, inter

    def PrimitiveIntersect(self, prim, o, d):
        """Primitive::Intersect of primitive `prim` (final order)."""
        o, d = _c3(o), _c3(d)
        n = o.shape[0]
        hit = np.zeros(n, np.int32)
        t = np.zeros(n, np.float32)
        nrm = np.zeros((n, 3), np.float32)
        inter = np.zeros(n, np.int32)
        _check(self.lib, self.lib.rtc_primitive_intersect(self.h, prim, n, o, d, hit, t, nrm, inter))
        return hit, t, nrm, inter

    def ToUInts(self, rgb):
        """AcesTonemap + GammaCorrected + Color::toUInts."""
        rgb = np.ascontiguousarray(rgb, np.float32).reshape(-1, 3)
        out = np.zeros(rgb.shape, np.uint8)
        _check(self.lib, self.lib.rtc_tonemap_u8(self.h, rgb.shape[0], rgb, out))
        return out

    def RenderSum(self, seed=0, sample_begin=0, sample_count=None):
        """Linear per-pixel radiance sums over a sample range, as an (H, W, 3) host array."""
        if sample_count is None:
            # hw1 / hw2 have no SAMPLES word: their one deterministic frame is "sample 0"
            sample_count = 1 if self.dialect <= 2 else self.samples
        out = np.zeros((self.height, self.width, 3), np.float32)
        _check(self.lib, self.lib.rtc_render_sum(self.h, seed, sample_begin, sample_count, out))
        return out

    def Render(self, seed=0):
        """Scene::Render: the tonemapped 8-bit image as an (H, W, 3) host array."""
        out = np.zeros((self.height, self.width, 3), np.uint8)
        _check(self.lib, self.lib.rtc_render_u8(self.h, seed, out))
        return out

    def RenderAdaptive(self, tolerance, min_samples=16, max_samples=0, seed=0):
        """Scene::Render with a noise threshold (rtc_render_adaptive): each 8x8 tile takes samples until the difference
        between the means of its even and its odd samples, in display units, is below `tolerance`, at most
        `max_samples` (0 = the scene's SAMPLES).  Returns the 8-bit image (H, W, 3), the even / odd sample sums
        (H, W, 2, 3 float32), the samples per pixel (H, W uint32) and the stats dict (passes, paths, tiles,
        tiles_stopped)."""
        img = np.zeros((self.height, self.width, 3), np.uint8)
        halves = np.zeros((self.height, self.width, 2, 3), np.float32)
        spp = np.zeros((self.height, self.width), np.uint32)
        st = np.zeros(4, np.uint64)
        _check(self.lib, self.lib.rtc_render_adaptive(self.h, seed, float(tolerance), min_samples, max_samples,
                                                      img, halves, spp, st))
        return img, halves, spp, dict(zip(["passes", "paths", "tiles", "tiles_stopped"], [int(v) for v in st]))

    def RenderAdaptiveMulti(self, devices, tolerance, min_samples=16, max_samples=0, seed=0):
        """RenderAdaptive on several CUDA devices of this process (rtc_render_adaptive_multi): tile t is rendered by
        devices[t % len(devices)], and devices[0] gathers the image over peer access.  Returns what RenderAdaptive
        returns; stats["passes"] is the most passes of any device."""
        dv = np.asarray(devices, np.int32)
        img = np.zeros((self.height, self.width, 3), np.uint8)
        halves = np.zeros((self.height, self.width, 2, 3), np.float32)
        spp = np.zeros((self.height, self.width), np.uint32)
        st = np.zeros(4, np.uint64)
        _check(self.lib, self.lib.rtc_render_adaptive_multi(self.h, dv, len(dv), seed, float(tolerance), min_samples,
                                                            max_samples, img, halves, spp, st))
        return img, halves, spp, dict(zip(["passes", "paths", "tiles", "tiles_stopped"], [int(v) for v in st]))

    def Denoise(self, halves, spp, strength=DENOISE_STRENGTH):
        """Non-local-means filter (rtc_denoise) on the (H, W, 2, 3) half sums and (H, W) samples per pixel that
        RenderAdaptive / RenderAdaptiveMulti return; every pixel needs at least 2 samples.  Returns the 8-bit image
        (H, W, 3) and the filtered linear mean (H, W, 3 float32); strength 0 returns the unfiltered image."""
        halves = np.ascontiguousarray(halves, np.float32)
        spp = np.ascontiguousarray(spp, np.uint32)
        if halves.shape != (self.height, self.width, 2, 3) or spp.shape != (self.height, self.width):
            raise ValueError("expected halves (%d, %d, 2, 3) and spp (%d, %d), got %s and %s"
                             % (self.height, self.width, self.height, self.width, halves.shape, spp.shape))
        img = np.zeros((self.height, self.width, 3), np.uint8)
        mean = np.zeros((self.height, self.width, 3), np.float32)
        _check(self.lib, self.lib.rtc_denoise(self.h, halves.ctypes.data_as(C.c_void_p), spp.ctypes.data_as(C.c_void_p),
                                              float(strength), img, mean.ctypes.data_as(C.c_void_p)))
        return img, mean

    def RenderDenoised(self, strength=DENOISE_STRENGTH, tolerance=0.0, min_samples=None, max_samples=0, seed=0):
        """RenderAdaptive's passes, then the filter of Denoise on the half sums where they lie (rtc_render_denoised).
        min_samples=None renders every pixel at the maximum (max_samples, or the scene's SAMPLES when it is 0).  Returns
        the 8-bit image (H, W, 3), the filtered mean (H, W, 3 float32) and RenderAdaptive's stats dict."""
        if min_samples is None:
            min_samples = max(2, max_samples or self.samples)
        img = np.zeros((self.height, self.width, 3), np.uint8)
        mean = np.zeros((self.height, self.width, 3), np.float32)
        st = np.zeros(4, np.uint64)
        _check(self.lib, self.lib.rtc_render_denoised(self.h, seed, float(tolerance), min_samples, max_samples, float(strength),
                                                      img, mean.ctypes.data_as(C.c_void_p), st))
        return img, mean, dict(zip(["passes", "paths", "tiles", "tiles_stopped"], [int(v) for v in st]))

    def RenderDenoisedMulti(self, devices, strength=DENOISE_STRENGTH, tolerance=0.0, min_samples=None, max_samples=0, seed=0):
        """RenderDenoised on several CUDA devices of this process (rtc_render_denoised_multi): RenderAdaptiveMulti's
        passes, then every entry filters a band of rows where the half sums lie.  min_samples=None means what it means
        for RenderDenoised.  Returns the 8-bit image (H, W, 3), the filtered mean (H, W, 3 float32), the half sums
        (H, W, 2, 3 float32) and samples per pixel (H, W uint32) the filter read, and RenderAdaptiveMulti's stats dict."""
        if min_samples is None:
            min_samples = max(2, max_samples or self.samples)
        dv = np.asarray(devices, np.int32)
        img = np.zeros((self.height, self.width, 3), np.uint8)
        mean = np.zeros((self.height, self.width, 3), np.float32)
        halves = np.zeros((self.height, self.width, 2, 3), np.float32)
        spp = np.zeros((self.height, self.width), np.uint32)
        st = np.zeros(4, np.uint64)
        _check(self.lib, self.lib.rtc_render_denoised_multi(self.h, dv, len(dv), seed, float(tolerance), min_samples, max_samples,
                                                            float(strength), img, mean.ctypes.data_as(C.c_void_p),
                                                            halves.ctypes.data_as(C.c_void_p), spp.ctypes.data_as(C.c_void_p), st))
        return img, mean, halves, spp, dict(zip(["passes", "paths", "tiles", "tiles_stopped"], [int(v) for v in st]))

    def RenderMulti(self, devices, seed=0, want_sum=False):
        """Scene::Render on several CUDA devices of this process: samples split over `devices`, summed over peer
        access and resolved on devices[0].  Returns the 8-bit image (and the float sums with want_sum)."""
        dv = np.asarray(devices, np.int32)
        out = np.zeros((self.height, self.width, 3), np.uint8)
        total = np.zeros((self.height, self.width, 3), np.float32) if want_sum else None
        _check(self.lib, self.lib.rtc_render_u8_multi(self.h, dv, len(dv), seed, out,
                                                      total.ctypes.data_as(C.c_void_p) if want_sum else None))
        return (out, total) if want_sum else out

    def arena_check(self):
        """Bytes of the scene arena in HBM that differ from the arena the host would have uploaded in full."""
        n = np.zeros(1, np.uint64)
        _check(self.lib, self.lib.rtc_scene_arena_check(self.h, n))
        return int(n[0])

    def upload_async(self):
        """Queue the H2D copy of the flattened scene into the arena that is not being read; the next render waits for it."""
        n = np.zeros(1, np.uint64)
        _check(self.lib, self.lib.rtc_scene_upload_async(self.h, n))
        return int(n[0])

    def frame_begin(self, seed=0, slot=0):
        """Queue one whole frame (scene upload, render, resolve, image to a pinned host buffer); returns the H2D bytes."""
        n = np.zeros(1, np.uint64)
        _check(self.lib, self.lib.rtc_frame_begin(self.h, seed, slot, n))
        return int(n[0])

    def frame_end(self, slot=0, out=None):
        """Wait for the frame of `slot`; copies the image into `out` (uint8, H x W x 3) when given."""
        _check(self.lib, self.lib.rtc_frame_end(self.h, slot, out.ctypes.data_as(C.c_void_p) if out is not None else None))
        return out

    def resolve_to_host(self, accum_ptr, total_samples, stream=None):
        _check(self.lib, self.lib.rtc_resolve_to_host_async(self.h, C.c_void_p(accum_ptr), total_samples, C.c_void_p(stream or 0)))

    def host_image_wait(self, out=None):
        _check(self.lib, self.lib.rtc_host_image_wait(self.h, out.ctypes.data_as(C.c_void_p) if out is not None else None))
        return out

    def intersect_dev(self, n, o_ptr, d_ptr, id_ptr, t_ptr, normal_ptr, interior_ptr, mode=0, stream=None):
        """Scene::RayIntersection on device arrays (pointers as integers), asynchronous on `stream`."""
        _check(self.lib, self.lib.rtc_intersect_dev(self.h, n, C.c_void_p(o_ptr), C.c_void_p(d_ptr), C.c_void_p(id_ptr),
                                                    C.c_void_p(t_ptr), C.c_void_p(normal_ptr), C.c_void_p(interior_ptr),
                                                    mode, C.c_void_p(stream or 0)))

    def RenderPPM(self, path, seed=0):
        _check(self.lib, self.lib.rtc_render_ppm(self.h, seed, os.fsencode(path)))

    def render_accumulate(self, accum_ptr, seed, sample_begin, sample_count, stream=None):
        """Device-pointer variant used by bench.py: adds into a float32 (H*W*3) device buffer."""
        _check(self.lib, self.lib.rtc_render_accumulate(self.h, seed, sample_begin, sample_count,
                                                         C.c_void_p(accum_ptr), C.c_void_p(stream or 0)))

    def render_resolve(self, accum_ptr, total_samples, rgb_ptr, stream=None):
        _check(self.lib, self.lib.rtc_render_resolve(self.h, C.c_void_p(accum_ptr), total_samples,
                                                      C.c_void_p(rgb_ptr), C.c_void_p(stream or 0)))

    def counters(self, stream=None):
        out = np.zeros(8, np.uint64)
        _check(self.lib, self.lib.rtc_render_counters(self.h, C.c_void_p(stream or 0), out))
        keys = ["paths", "rays", "launches", "batches", "index_node_visits", "fallback_rays", "prim_tests", "traversed_rays"]
        return dict(zip(keys, [int(v) for v in out[:8]]))

    def traverse_lanes(self, stream=None):
        """Warp-execution efficiency of k_traverse's scheduler (needs set_profiling(count_visits=True)): per kind
        (visit, leaf, finish, refill) the warp iterations and the mean number of lanes (of 32) that took part."""
        out = np.zeros(8, np.uint64)
        _check(self.lib, self.lib.rtc_traverse_lanes(self.h, C.c_void_p(stream or 0), out))
        kinds = ["visit", "leaf", "finish", "refill"]
        return {k: {"iterations": int(out[i]), "lanes": (float(out[4 + i]) / float(out[i]) if out[i] else 0.0)}
                for i, k in enumerate(kinds)}

    def set_profiling(self, kernel_events=False, count_visits=False):
        _check(self.lib, self.lib.rtc_set_profiling(self.h, int(kernel_events), int(count_visits)))

    def profile(self, stream=None, reset=True):
        """Per kernel class (generate, traverse, shade, pre): total ms and launches."""
        ms = np.zeros(4, np.float64)
        n = np.zeros(4, np.uint64)
        _check(self.lib, self.lib.rtc_render_profile(self.h, C.c_void_p(stream or 0), ms, n, int(reset)))
        names = ["generate", "traverse", "shade", "pre"]
        return {k: {"ms": float(ms[i]), "launches": int(n[i])} for i, k in enumerate(names)}

    def reset_counters(self):
        _check(self.lib, self.lib.rtc_render_reset_counters(self.h))


def shard_samples(samples, rank, world):
    """spp sharding of Scene::Sample's loop over `world` ranks: rank r renders samples
    [lo, hi).  Ranges are disjoint, cover [0, samples) and differ in size by at most one."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError("bad rank/world")
    return rank * samples // world, (rank + 1) * samples // world


def philox4x32_10(ctr, key):
    out = np.zeros(4, np.uint32)
    load_library().rtc_philox4x32_10(np.asarray(ctr, np.uint32), np.asarray(key, np.uint32), out)
    return out
