"""Adaptive sampling on several devices (rtc_render_adaptive_multi / Scene.RenderAdaptiveMulti): tile t of the frame is
rendered by devices[t % len(devices)] with the pass loop of rtc_render_adaptive, and devices[0] gathers the image.

A tile's decisions read only its own half sums and the RNG is a pure function of (seed, pixel, sample, bounce), so the
result is the one-device call's up to float summation order.  Each check compares against RenderSum, the one-device
RenderAdaptive and the numpy model of the rule in test_adaptive.py.  On a one-GPU machine a device is listed several
times: each entry is a replica of the scene with its own buffers and stream, which runs the whole path."""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import scene_path
from test_adaptive import TILE, half_sums, model, per_tile, tile_errors
from test_dialects import load as load_dialect


def _devices(rtc, n):
    """n entries over the first two devices when the box has two, else device 0 n times"""
    k = 2 if rtc.device_count() >= 2 else 1
    return [i % k for i in range(n)]


def _close(got, want):
    ok = np.isfinite(got) & np.isfinite(want)
    assert ok.mean() > 0.999
    assert np.allclose(got[ok], want[ok], rtol=1e-4, atol=1e-5), np.abs(got[ok] - want[ok]).max()


def _schedule(s, nmin, smax, seed):
    """Per-sample images of `s`, a tau that leaves at least two sample counts in the model, the model's per-tile
    counts and each tile's margin |E - tau| over its decisions"""
    samples = np.stack([s.RenderSum(seed=seed, sample_begin=k, sample_count=1) for k in range(smax)])
    A, B = samples[0:nmin:2].sum(0, dtype=np.float32), samples[1:nmin:2].sum(0, dtype=np.float32)
    e0 = tile_errors(A, B, nmin)
    levels = 3 if e0.size >= 16 else 2
    for q in (0.5, 0.4, 0.6, 0.3, 0.7, 0.2, 0.8):
        tau = float(np.float32(np.quantile(e0, q)))   # the library takes tau as a float
        if tau > 0 and len(np.unique(model(samples, tau, nmin, smax)[0])) >= levels:
            want_n, margin = model(samples, tau, nmin, smax)
            return samples, tau, want_n, margin
    raise AssertionError("no tau with %d sample-count levels" % levels)


def _matches_one_device(s, devices, nmin, smax, seed):
    samples, tau, want_n, margin = _schedule(s, nmin, smax, seed)
    img, halves, spp, st = s.RenderAdaptiveMulti(devices, tau, min_samples=nmin, max_samples=smax, seed=seed)
    img1, halves1, spp1, st1 = s.RenderAdaptive(tau, min_samples=nmin, max_samples=smax, seed=seed)
    got_n, one_n = spp[::TILE, ::TILE], spp1[::TILE, ::TILE]
    clear = margin > 1e-3 * tau + 1e-6
    assert clear.any()
    assert np.array_equal(got_n[clear], want_n[clear]), np.argwhere(got_n != want_n)
    assert np.array_equal(got_n[clear], one_n[clear])
    assert (per_tile(got_n, s.height, s.width) == spp).all()   # one count per tile
    assert st["paths"] == int(spp.sum())
    assert st["tiles"] == want_n.size and st["tiles_stopped"] == int((got_n < smax).sum())
    A, B = half_sums(samples, spp)
    _close(halves[:, :, 0], A)
    _close(halves[:, :, 1], B)
    same = spp == spp1
    assert (np.abs(img[same].astype(int) - img1[same].astype(int)) <= 1).mean() >= 0.999
    return spp, st


# ---------------------------------------------------------------------------------------------- CPU
def test_adaptive_multi_binding_is_declared(rtc):
    assert "rtc_render_adaptive_multi" in rtc.exported_symbols()
    with open(rtc.HEADER_PATH) as f:
        assert "int rtc_render_adaptive_multi(" in f.read()
    assert callable(rtc.load_library().rtc_render_adaptive_multi)


@pytest.mark.parametrize("tolerance,min_samples,devices", [
    (float("nan"), 16, [0]), (float("inf"), 16, [0]), (-1.0 / 255, 16, [0]), (0.01, 1, [0]), (0.01, 0, [0]),
    (0.01, 16, []), (0.01, 16, [0] * 17), (0.01, 16, [64]), (0.01, 16, [-1]), (0.01, 16, [0, 0, 64]),
])
def test_adaptive_multi_bad_arguments(rtc, tolerance, min_samples, devices):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.RenderAdaptiveMulti(devices, tolerance, min_samples=min_samples)
    s.close()


def _raw(rtc):
    """the entry point with plain pointers, so that null arguments can be passed"""
    f = C.CDLL(rtc.LIB_PATH).rtc_render_adaptive_multi
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                  C.c_void_p, C.c_void_p]
    return f


def test_adaptive_multi_null_scene_and_devices(rtc):
    f = _raw(rtc)
    dv = np.zeros(2, np.int32)
    assert f(None, dv.ctypes.data_as(C.c_void_p), 2, 0, 0.01, 16, 0, None, None, None, None) == -4
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    assert f(s.h, None, 2, 0, 0.01, 16, 0, None, None, None, None) == -4
    s.close()


def test_adaptive_multi_host_only_scene_has_no_fallback(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    with pytest.raises(rtc.RtcError, match="rtc error -2"):
        s.RenderAdaptiveMulti([0, 0], 0.01, min_samples=4)
    s.close()


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("entries", [2, 3, 5])
@pytest.mark.parametrize("name,w,h,spp", [("lights_mix", 96, 64, 16), ("practice5_dragon_10k", 128, 128, 8)])
def test_tolerance_zero_is_the_full_render(rtc, name, w, h, spp, entries):
    s = rtc.Scene(path=scene_path(name), device=0)
    s.override(w, h, spp)
    img, halves, n, st = s.RenderAdaptiveMulti(_devices(rtc, entries), 0.0, min_samples=2, seed=4)
    assert (n == spp).all()
    assert st["paths"] == w * h * spp
    assert st["tiles"] == math.ceil(w / 8) * math.ceil(h / 8) and st["tiles_stopped"] == 0
    assert st["passes"] == 1 + int(math.log2(spp // 2))
    _close(halves.sum(2), s.RenderSum(seed=4, sample_begin=0, sample_count=spp))
    ref = s.Render(seed=4)
    assert (np.abs(img.astype(int) - ref.astype(int)) <= 1).mean() >= 0.999
    s.close()


@pytest.mark.gpu
def test_schedule_matches_the_numpy_model_and_one_device(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(60, 44, 64)
    spp, st = _matches_one_device(s, _devices(rtc, 3), 4, 64, 17)
    s.close()
    assert len(np.unique(spp)) >= 3


@pytest.mark.gpu
def test_more_devices_than_tiles(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(16, 8, 32)
    _matches_one_device(s, _devices(rtc, 3), 2, 32, 9)
    img, halves, spp, st = s.RenderAdaptiveMulti(_devices(rtc, 3), 0.0, min_samples=2, seed=9)
    s.close()
    assert (spp == 32).all() and st["tiles"] == 2 and st["paths"] == 16 * 8 * 32


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0], [1, 0]])
def test_one_entry_and_a_head_that_is_not_the_scene_device(rtc, devices):
    if max(devices) >= rtc.device_count():
        pytest.skip("needs %d devices" % (max(devices) + 1))
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(60, 44, 64)
    _matches_one_device(s, devices, 4, 64, 21)
    s.close()


@pytest.mark.gpu
def test_empty_frame(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(0, 0, 16)
    img, halves, spp, st = s.RenderAdaptiveMulti(_devices(rtc, 2), 0.01)
    s.close()
    assert img.size == 0 and st == {"passes": 0, "paths": 0, "tiles": 0, "tiles_stopped": 0}


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw1_course_sample6", "hw2_hw2_lights"])
def test_deterministic_dialects_render_their_one_frame(rtc, fixture):
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    want = s.RenderAdaptive(0.01, min_samples=4, seed=3)
    got = s.RenderAdaptiveMulti(_devices(rtc, 2), 0.01, min_samples=4, seed=3)
    s.close()
    for a, b in zip(got[:3], want[:3]):
        assert np.array_equal(a, b)
    assert got[3] == want[3] and (got[2] == 1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw3_course_sample3", "hw4_course_sample3"])
def test_monte_carlo_dialects_at_tolerance_zero(rtc, fixture):
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    spp = min(s.samples, 16)
    s.override(-1, -1, spp)
    img, halves, n, st = s.RenderAdaptiveMulti(_devices(rtc, 3), 0.0, min_samples=2, seed=8)
    want = s.RenderSum(seed=8, sample_begin=0, sample_count=spp)
    s.close()
    assert (n == spp).all()
    _close(halves.sum(2), want)


@pytest.mark.gpu
def test_no_interference_with_the_other_render_paths(rtc):
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=0)
    s.override(160, 120, 8)
    devices = _devices(rtc, 2)
    before = s.RenderSum(seed=12, sample_count=8)
    want = [s.Render(seed=30 + i) for i in range(2)]
    multi = s.RenderMulti(devices, seed=30)
    s.RenderAdaptiveMulti(devices, 2 / 255, min_samples=2, seed=12)
    _close(s.RenderSum(seed=12, sample_count=8), before)
    assert (np.abs(s.Render(seed=30).astype(int) - want[0].astype(int)) <= 1).mean() > 0.999
    got = [np.zeros_like(want[0]) for _ in range(2)]
    s.frame_begin(seed=30, slot=0)
    s.frame_begin(seed=31, slot=1)
    s.frame_end(0, got[0])
    s.frame_end(1, got[1])
    for a, b in zip(want, got):
        assert (np.abs(a.astype(int) - b.astype(int)) <= 1).mean() > 0.999
    again = s.RenderMulti(devices, seed=30)
    s.close()
    assert (np.abs(again.astype(int) - multi.astype(int)) <= 1).mean() > 0.999
