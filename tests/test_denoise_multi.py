"""Denoising on several devices (rtc_render_denoised_multi / Scene.RenderDenoisedMulti): the passes of
RenderAdaptiveMulti, then entry i of the device list filters the image rows of the tile rows [i T / n, (i + 1) T / n) of
the filter's grid (T = ceil(H / 16)), reading those rows and APRON more on either side from the tiles' owners.

The bands together are the one-device grid block for block, so the call's image and mean equal those of Denoise on the
half sums and spp that the same call returns, bit for bit.  Two calls do not agree to the bit (the render's float
atomics), which is why the call returns the half sums it filtered.  On a one-GPU machine a device is listed several
times (test_adaptive_multi._devices): each entry is a replica of the scene with its own buffers and stream."""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import scene_path
from test_adaptive_multi import _devices
from test_denoise import F, R, S, nlm, synthetic
from test_dialects import load as load_dialect

TILE_H = 16              # rt_kernels.h kDenoiseTileH
APRON = R + F + S        # rows beyond its band that an entry reads (rt_kernels.h kDenoiseApron)


def bands(h, n):
    """(y0, y1) of every entry: the output rows of its tile rows"""
    t = -(-h // TILE_H)
    return [(TILE_H * (i * t // n), min(h, TILE_H * ((i + 1) * t // n))) for i in range(n)]


def _raw(rtc):
    """the entry point with plain pointers, so that null arguments can be passed"""
    f = C.CDLL(rtc.LIB_PATH).rtc_render_denoised_multi
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_float, C.c_uint32, C.c_uint32, C.c_float, C.c_void_p,
                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return f


# ---------------------------------------------------------------------------------------------- CPU
def test_denoise_multi_binding_is_declared(rtc):
    assert "rtc_render_denoised_multi" in rtc.exported_symbols()
    with open(rtc.HEADER_PATH) as f:
        assert "int rtc_render_denoised_multi(" in f.read()
    assert callable(rtc.load_library().rtc_render_denoised_multi)


@pytest.mark.parametrize("kw,devices", [
    (dict(strength=float("nan")), [0]), (dict(strength=float("inf")), [0]), (dict(strength=-0.5), [0]),
    (dict(tolerance=float("nan")), [0]), (dict(tolerance=float("inf")), [0]), (dict(tolerance=-1 / 255), [0]),
    (dict(min_samples=1), [0]), (dict(min_samples=0), [0]), (dict(min_samples=2, max_samples=1), [0]),
    ({}, []), ({}, [0] * 17), ({}, [64]), ({}, [-1]), ({}, [0, 0, 64]),
])
def test_denoise_multi_bad_arguments(rtc, kw, devices):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.RenderDenoisedMulti(devices, **kw)
    s.close()


def test_denoise_multi_null_scene_and_devices(rtc):
    f = _raw(rtc)
    dv = np.zeros(2, np.int32)
    assert f(None, dv.ctypes.data_as(C.c_void_p), 2, 0, 0.0, 16, 0, 0.45, None, None, None, None, None) == -4
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    assert f(s.h, None, 2, 0, 0.0, 16, 0, 0.45, None, None, None, None, None) == -4
    s.override(-1, -1, 1)   # a maximum of 1 sample from SAMPLES
    assert f(s.h, dv.ctypes.data_as(C.c_void_p), 2, 0, 0.0, 2, 0, 0.45, None, None, None, None, None) == -4
    s.close()


def test_denoise_multi_host_only_scene_has_no_fallback(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    for call in (lambda: s.RenderDenoisedMulti([0, 0]), lambda: s.RenderDenoisedMulti([0], 0.0, tolerance=0.01, min_samples=4)):
        with pytest.raises(rtc.RtcError, match="rtc error -2"):
            call()
    s.close()


@pytest.mark.parametrize("w,h,n", [(61, 37, 2), (61, 37, 3), (96, 20, 5), (1, 1, 3), (200, 3, 2), (24, 70, 4), (9, 50, 8)])
def test_bands_reproduce_the_whole_frame(w, h, n):
    """the rule in numpy: the filter of each entry's prep rows, cut to its output rows, is the filter of the whole frame"""
    halves, spp = synthetic(w, h, 31 + w + h + n, nonfinite=False)
    for k in (0.45, 1.0):
        whole = nlm(halves, spp, k)
        got = np.full_like(whole, np.nan)
        for y0, y1 in bands(h, n):
            if y0 == y1:
                continue
            r0, r1 = max(0, y0 - APRON), min(h, y1 + APRON)
            got[y0:y1] = nlm(halves[r0:r1], spp[r0:r1], k)[y0 - r0:y1 - r0]
        # equal up to the float64 rounding of the model's running sums, which start at another row
        assert np.allclose(got, whole, rtol=1e-9, atol=1e-12), (k, np.abs(got - whole).max())
    covered = [y for y0, y1 in bands(h, n) for y in range(y0, y1)]
    assert covered == list(range(h))   # every row once, in order
    assert sum(y0 == y1 for y0, y1 in bands(h, n)) == max(0, n - math.ceil(h / TILE_H))


# ---------------------------------------------------------------------------------------------- GPU
def _exact(s, devices, k, **kw):
    """RenderDenoisedMulti against Denoise on the half sums and spp of the same call, bit for bit"""
    img, mean, halves, spp, st = s.RenderDenoisedMulti(devices, k, **kw)
    img1, mean1 = s.Denoise(halves, spp, k)
    assert np.array_equal(mean, mean1, equal_nan=True), np.argwhere(~((mean == mean1) | (np.isnan(mean) & np.isnan(mean1))))[:5]
    assert np.array_equal(img, img1)
    return img, mean, halves, spp, st


@pytest.mark.gpu
@pytest.mark.parametrize("entries", [1, 2, 3, 5, 8])
def test_bands_are_the_one_device_filter(rtc, entries):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(72, 100, 8)   # 7 tile rows of the filter: 8 entries leave one without a band
    for k in (rtc.DENOISE_STRENGTH, 1.0):
        _, _, halves, spp, st = _exact(s, _devices(rtc, entries), k, seed=3)
        assert (spp == 8).all() and st["paths"] == 72 * 100 * 8 and st["tiles"] == 9 * 13
        want = s.RenderSum(seed=3, sample_count=8)
        ok = np.isfinite(want)
        assert np.allclose(halves.sum(2)[ok], want[ok], rtol=1e-4, atol=1e-5)
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,entries", [(61, 37, 3), (96, 20, 5), (1, 1, 2), (200, 3, 3)])
def test_frame_shapes(rtc, w, h, entries):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(w, h, 8)
    for k in (rtc.DENOISE_STRENGTH, 1.0):
        _exact(s, _devices(rtc, entries), k, seed=5)
    s.close()


@pytest.mark.gpu
def test_stopped_tiles_across_band_edges(rtc):
    s = rtc.Scene(path=scene_path("practice5_1"), device=0)
    s.override(80, 72, 32)
    for k in (rtc.DENOISE_STRENGTH, 1.0):
        _, _, _, spp, st = _exact(s, _devices(rtc, 3), k, tolerance=2 / 255, min_samples=4, max_samples=32, seed=6)
        assert st["tiles_stopped"] > 0 and len(np.unique(spp)) >= 2
        # the bands of 3 entries start at rows 16 and 48: spp changes across at least one of those edges somewhere
        assert any((spp[y - 1] != spp[y]).any() for y0, _ in bands(72, 3)[1:] for y in [y0])
    s.close()


@pytest.mark.gpu
def test_at_4k(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(3840, 2160, 8)
    _exact(s, _devices(rtc, 8), rtc.DENOISE_STRENGTH, seed=2)
    s.close()


@pytest.mark.gpu
def test_strength_zero_is_the_unfiltered_image(rtc):
    s = rtc.Scene(path=scene_path("practice5_1"), device=0)
    s.override(80, 56, 32)
    img, mean, halves, spp, _ = s.RenderDenoisedMulti(_devices(rtc, 3), 0.0, tolerance=2 / 255, min_samples=4, seed=6)
    assert len(np.unique(spp)) >= 2
    want = (halves[:, :, 0] + halves[:, :, 1]) * (np.float32(1) / spp.astype(np.float32))[:, :, None]
    assert np.array_equal(mean, want, equal_nan=True)
    assert np.array_equal(img.reshape(-1, 3), s.ToUInts(want.reshape(-1, 3)))
    s.close()


@pytest.mark.gpu
def test_agrees_with_the_one_device_call(rtc):
    s = rtc.Scene(path=scene_path("practice5_1"), device=0)
    s.override(128, 96, 16)
    k = rtc.DENOISE_STRENGTH
    img, mean, _, _, st = s.RenderDenoisedMulti(_devices(rtc, 3), k, seed=21)
    img1, mean1, st1 = s.RenderDenoised(k, seed=21)
    s.close()
    assert st == st1
    close = np.isclose(mean, mean1, rtol=1e-3, atol=1e-6) | (np.isnan(mean) & np.isnan(mean1))
    assert close.mean() >= 0.999
    assert (np.abs(img.astype(int) - img1.astype(int)) <= 1).mean() >= 0.999


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw1_course_sample6", "hw2_hw2_lights"])
def test_deterministic_dialects_are_not_filtered(rtc, fixture):
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    img, mean, halves, spp, st = s.RenderDenoisedMulti(_devices(rtc, 2), 1.0, seed=3)
    want_img, want_mean, want_st = s.RenderDenoised(1.0, seed=3)
    s.close()
    assert np.array_equal(img, want_img) and np.array_equal(mean, want_mean) and st == want_st
    assert (spp == 1).all() and np.array_equal(halves[:, :, 0], want_mean) and (halves[:, :, 1] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw3_course_sample3", "hw4_course_sample3"])
def test_monte_carlo_dialects_at_strength_zero_are_the_render(rtc, fixture):
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    s.override(-1, -1, min(s.samples, 16))
    img = s.RenderDenoisedMulti(_devices(rtc, 3), 0.0, seed=9)[0]
    ref = s.Render(seed=9)
    s.close()
    assert (np.abs(img.astype(int) - ref.astype(int)) <= 1).mean() >= 0.999


@pytest.mark.gpu
def test_no_interference_with_the_other_render_paths(rtc):
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=0)
    s.override(160, 120, 8)
    devices = _devices(rtc, 3)
    before = s.RenderSum(seed=12, sample_count=8)
    want = [s.Render(seed=30 + i) for i in range(2)]
    multi = s.RenderMulti(devices, seed=30)
    _, ad_halves, ad_spp, _ = s.RenderAdaptiveMulti(devices, 0.0, min_samples=2, seed=12)
    dn_img, dn_mean, _ = s.RenderDenoised(seed=12)
    s.RenderDenoisedMulti(devices, seed=12)
    s.RenderDenoisedMulti(devices, 0.0, tolerance=2 / 255, min_samples=2, seed=12)
    after = s.RenderSum(seed=12, sample_count=8)
    ok = np.isfinite(before) & np.isfinite(after)
    assert np.allclose(before[ok], after[ok], rtol=1e-4, atol=1e-5)
    assert [(np.abs(s.Render(seed=30 + i).astype(int) - a.astype(int)) <= 1).mean() > 0.999 for i, a in enumerate(want)] == [True, True]
    got = [np.zeros_like(want[0]) for _ in range(2)]
    s.frame_begin(seed=30, slot=0)
    s.frame_begin(seed=31, slot=1)
    s.frame_end(0, got[0])
    s.frame_end(1, got[1])
    for a, b in zip(want, got):
        assert (np.abs(a.astype(int) - b.astype(int)) <= 1).mean() > 0.999
    assert (np.abs(s.RenderMulti(devices, seed=30).astype(int) - multi.astype(int)) <= 1).mean() > 0.999
    _, halves, spp, _ = s.RenderAdaptiveMulti(devices, 0.0, min_samples=2, seed=12)
    assert np.array_equal(spp, ad_spp)
    ok = np.isfinite(halves) & np.isfinite(ad_halves)
    assert np.allclose(halves[ok], ad_halves[ok], rtol=1e-4, atol=1e-5)
    img, mean, _ = s.RenderDenoised(seed=12)
    s.close()
    close = np.isclose(mean, dn_mean, rtol=1e-3, atol=1e-6) | (np.isnan(mean) & np.isnan(dn_mean))
    assert close.mean() >= 0.999
    assert (np.abs(img.astype(int) - dn_img.astype(int)) <= 1).mean() >= 0.999


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0, 1, 0], [1, 0]])
def test_two_gpus_and_a_head_that_is_not_the_scene_device(rtc, devices):
    if rtc.device_count() < 2:
        pytest.skip("needs 2 devices")
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(96, 80, 16)
    for k in (rtc.DENOISE_STRENGTH, 1.0):
        _exact(s, devices, k, tolerance=2 / 255, min_samples=4, seed=8)
    s.close()
