"""Denoising (rtc_denoise / Scene.Denoise, rtc_render_denoised / Scene.RenderDenoised): non-local means on the even /
odd half sums of a render, with their difference as the per-pixel noise estimate (DESIGN.md "Denoising").

The kernels are checked against `nlm`, a numpy restatement of the rule, on synthetic half sums; the entry points against
the renders they are made of; the quality against our own render at many samples."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, scene_path
from test_adaptive import aces, display, squash
from test_dialects import load as load_dialect

# the fixed constants of the rule (rt_kernels.h kDenoise*): window (2R+1)^2, patch (2F+1)^2, the box (2S+1)^2 that
# smooths V, alpha, epsilon
R, F, S, ALPHA, EPS = 7, 3, 1, 1.0, 1e-8


# ---------------------------------------------------------------------------------------------- the rule in numpy
def prep(halves, spp):
    """u, D, V of k_denoise_prep (float32, the kernel's operations) from (H, W, 2, 3) halves and (H, W) spp"""
    n = spp.astype(np.float32)[:, :, None]
    A, B = halves[:, :, 0], halves[:, :, 1]
    with np.errstate(invalid="ignore", over="ignore"):
        u = (np.float32(1) / n) * (A + B)
        ia = np.float32(1) / ((spp + 1) // 2).astype(np.float32)[:, :, None]
        ib = np.float32(1) / (spp // 2).astype(np.float32)[:, :, None]
        e = (display(A * ia) - display(B * ib)) * np.float32(0.5)
    return u.astype(np.float32), display(u), (e * e).astype(np.float32)


def nlm(halves, spp, k):
    """The filtered mean of every pixel (float64); k = 0 is the identity"""
    u, D, V = prep(halves, spp)
    if k == 0:
        return u
    h, w = spp.shape
    Vb = np.pad(V.astype(np.float64), ((S, S), (S, S), (0, 0)), mode="edge")
    V = sum(Vb[oy:oy + h, ox:ox + w] for oy in range(2 * S + 1) for ox in range(2 * S + 1)) / (2 * S + 1) ** 2
    A_ = R + F
    Dp = np.pad(D.astype(np.float64), ((A_, A_), (A_, A_), (0, 0)), mode="edge")   # patches repeat the edge pixels
    Vp = np.pad(V, ((A_, A_), (A_, A_), (0, 0)), mode="edge")
    up = np.pad(u.astype(np.float64), ((R, R), (R, R), (0, 0)), constant_values=np.nan)   # outside: not a neighbour
    eh, ew = h + 2 * F, w + 2 * F
    d0, v0 = Dp[R:R + eh, R:R + ew], Vp[R:R + eh, R:R + ew]
    sw = np.zeros((h, w))
    su = np.zeros((h, w, 3))
    for dy in range(-R, R + 1):
        for dx in range(-R, R + 1):
            d1, v1 = Dp[R + dy:R + dy + eh, R + dx:R + dx + ew], Vp[R + dy:R + dy + eh, R + dx:R + dx + ew]
            t = (((d0 - d1) ** 2 - ALPHA * (v0 + np.minimum(v0, v1))) / (EPS + k * k * (v0 + v1))).sum(2)
            c = np.pad(t.cumsum(0).cumsum(1), ((1, 0), (1, 0)))
            p = 2 * F + 1
            box = c[p:, p:] - c[:-p, p:] - c[p:, :-p] + c[:-p, :-p]
            wgt = np.exp(-np.maximum(0.0, box / (3 * p * p)))
            uq = up[R + dy:R + dy + h, R + dx:R + dx + w]
            ok = np.isfinite(uq).all(2)
            sw += np.where(ok, wgt, 0.0)
            su += np.where(ok[:, :, None], wgt[:, :, None] * np.nan_to_num(uq), 0.0)
    out = su / sw[:, :, None]
    bad = ~np.isfinite(u).all(2)
    out[bad] = u[bad]
    return out


def to_u8(x):
    return np.floor(np.float32(255) * display(np.asarray(x, np.float32)) + np.float32(0.5)).astype(np.uint8)


def synthetic(w, h, seed, nonfinite=True):
    """Half sums of a structured image (gradient, a step edge, a bright disc) with per-pixel noise at 2..64 spp"""
    rng = np.random.default_rng(seed)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([0.2 + 0.6 * xs / max(w, 1), 0.5 * (xs > w / 2), 0.1 + 0.3 * ys / max(h, 1)], 2)
    base[(xs - w / 3) ** 2 + (ys - h / 2) ** 2 < (min(w, h) / 4) ** 2] += 3.0
    spp = rng.integers(2, 65, (h, w)).astype(np.uint32)
    na, nb = ((spp + 1) // 2)[:, :, None].astype(np.float32), (spp // 2)[:, :, None].astype(np.float32)
    noisy = lambda n: np.abs(n * base + np.sqrt(n) * rng.normal(0, 0.5, base.shape)).astype(np.float32)
    halves = np.stack([noisy(na), noisy(nb)], 2).astype(np.float32)
    if nonfinite and w * h >= 8:
        flat = halves.reshape(-1, 2, 3)
        idx = rng.choice(w * h, max(1, w * h // 50), replace=False)
        flat[idx[0::2], 0, 0] = np.nan
        flat[idx[1::2], 1, 2] = np.inf
    return halves, spp


def host_scene(rtc, dialect_fixture=None):
    if dialect_fixture:
        text, dialect, _ = load_dialect(dialect_fixture)
        return rtc.Scene(text=text, device=-1, dialect=dialect)
    return rtc.Scene(path=scene_path("lights_mix"), device=-1)


# ---------------------------------------------------------------------------------------------- CPU
def test_denoise_bindings_are_declared(rtc):
    with open(rtc.HEADER_PATH) as f:
        header = f.read()
    for name in ("rtc_denoise", "rtc_render_denoised"):
        assert name in rtc.exported_symbols() and "int %s(" % name in header
        assert callable(getattr(rtc.load_library(), name))


@pytest.mark.parametrize("strength", [float("nan"), float("inf"), -0.5])
def test_bad_strength(rtc, strength):
    s = host_scene(rtc)
    halves = np.zeros((s.height, s.width, 2, 3), np.float32)
    spp = np.full((s.height, s.width), 4, np.uint32)
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.Denoise(halves, spp, strength)
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.RenderDenoised(strength)
    s.close()


def test_denoise_argument_errors_come_before_the_device(rtc):
    s = host_scene(rtc)
    halves = np.zeros((s.height, s.width, 2, 3), np.float32)
    spp = np.full((s.height, s.width), 4, np.uint32)
    spp[3, 5] = 1
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.Denoise(halves, spp)
    spp[3, 5] = 4
    img = np.zeros((s.height, s.width, 3), np.uint8)
    lib = s.lib
    assert lib.rtc_denoise(s.h, None, spp.ctypes.data_as(C.c_void_p), 0.5, img, None) == -4
    assert lib.rtc_denoise(s.h, halves.ctypes.data_as(C.c_void_p), None, 0.5, img, None) == -4
    with pytest.raises(ValueError):
        s.Denoise(halves[:, :-1], spp[:, :-1])
    for kw in (dict(tolerance=float("nan")), dict(tolerance=-1.0), dict(min_samples=1), dict(max_samples=1, min_samples=2)):
        with pytest.raises(rtc.RtcError, match="rtc error -4"):
            s.RenderDenoised(0.5, **kw)
    s.close()


@pytest.mark.parametrize("fixture", ["hw1_course_sample6", "hw2_hw2_lights"])
def test_deterministic_dialects_have_no_noise_to_filter(rtc, fixture):
    s = host_scene(rtc, fixture)
    halves = np.zeros((s.height, s.width, 2, 3), np.float32)
    spp = np.full((s.height, s.width), 4, np.uint32)
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.Denoise(halves, spp)
    s.close()


def test_denoise_has_no_cpu_fallback(rtc):
    s = host_scene(rtc)
    halves = np.ones((s.height, s.width, 2, 3), np.float32)
    spp = np.full((s.height, s.width), 4, np.uint32)
    for call in (lambda: s.Denoise(halves, spp), lambda: s.Denoise(halves, spp, 0.0), lambda: s.RenderDenoised(),
                 lambda: s.RenderDenoised(0.0, tolerance=0.01, min_samples=4)):
        with pytest.raises(rtc.RtcError, match="rtc error -2"):
            call()
    s.close()


def test_denoise_cli_rejects_bad_values(rtc, tmp_path):
    for value in ("abc", "-1", "nan"):
        env = dict(os.environ, RTC_DENOISE=value)
        r = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path("lights_mix"), str(tmp_path / "x.ppm")], env=env,
                           capture_output=True, text=True)
        assert r.returncode == 1, (value, r.stderr)
        assert "RTC_DENOISE" in r.stderr
    env = dict(os.environ, RTC_DENOISE="0.5", RTC_DEVICES="0,1")
    r = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path("lights_mix"), str(tmp_path / "x.ppm")], env=env,
                       capture_output=True, text=True)
    assert r.returncode == 1 and "RTC_DENOISE" in r.stderr


def test_numpy_model_of_the_rule():
    halves, spp = synthetic(24, 20, 1)
    u = prep(halves, spp)[0]
    assert np.array_equal(nlm(halves, spp, 0.0), u, equal_nan=True)
    # a flat grey image with noise: most of the error goes
    rng = np.random.default_rng(2)
    spp = np.full((24, 24), 8, np.uint32)
    flat = np.abs(4 * 0.3 + 2 * rng.normal(0, 0.3, (24, 24, 2, 3))).astype(np.float32)
    u = prep(flat, spp)[0]
    out = nlm(flat, spp, 0.45)
    assert np.sqrt(np.mean((out - 0.3) ** 2)) < 0.4 * np.sqrt(np.mean((u - 0.3) ** 2))
    # a noisy step edge keeps its step: the columns either side stay on their own level
    step = np.where(np.arange(24) < 12, 0.05, 0.8).astype(np.float32)[None, :, None, None]
    edge = np.abs(4 * step + 2 * rng.normal(0, 0.02, (24, 24, 2, 3))).astype(np.float32)
    out = nlm(edge, spp, 0.45)
    assert abs(out[:, 11].mean() - 0.05) < 0.02 and abs(out[:, 12].mean() - 0.8) < 0.05


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(61, 37), (1, 1), (1, 40), (200, 3)])
@pytest.mark.parametrize("k", ["default", 1.0])
def test_kernel_matches_the_numpy_model(rtc, w, h, k):
    k = rtc.DENOISE_STRENGTH if k == "default" else k
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(w, h, 8)
    halves, spp = synthetic(w, h, 10 + w + h)
    img, mean = s.Denoise(halves, spp, k)
    s.close()
    want = nlm(halves, spp, k)
    u = prep(halves, spp)[0]
    bad = ~np.isfinite(u).all(2)
    assert np.array_equal(mean[bad], u[bad], equal_nan=True)   # non-finite pixels pass through
    assert np.allclose(mean[~bad], want[~bad], rtol=1e-3, atol=1e-6), np.abs(mean[~bad] - want[~bad]).max()
    ref = to_u8(want)
    d = np.abs(img.astype(int) - ref.astype(int))[~bad]
    assert d.max() <= 1 and (d == 0).mean() >= 0.999


@pytest.mark.gpu
def test_strength_zero_is_the_unfiltered_image(rtc):
    s = rtc.Scene(path=scene_path("practice5_1"), device=0)
    s.override(80, 56, 32)
    _, halves, spp, _ = s.RenderAdaptive(2 / 255, min_samples=4, seed=6)
    assert len(np.unique(spp)) >= 2
    img, mean = s.Denoise(halves, spp, 0.0)
    want = (halves[:, :, 0] + halves[:, :, 1]) * (np.float32(1) / spp.astype(np.float32))[:, :, None]
    assert np.array_equal(mean, want, equal_nan=True)
    assert np.array_equal(img.reshape(-1, 3), s.ToUInts(want.reshape(-1, 3)))
    syn, sspp = synthetic(s.width, s.height, 4)
    img, mean = s.Denoise(syn, sspp, 0.0)
    want = prep(syn, sspp)[0]
    assert np.array_equal(mean, want, equal_nan=True)
    assert np.array_equal(img.reshape(-1, 3), s.ToUInts(want.reshape(-1, 3)))
    s.close()


def _fixture_scene(rtc, fixture):
    if fixture == "practice5_2":
        s = rtc.Scene(path=scene_path(fixture), device=0)
        s.override(96, 64, 16)
    else:
        text, dialect, _ = load_dialect(fixture)
        s = rtc.Scene(text=text, device=0, dialect=dialect)
        s.override(-1, -1, min(s.samples, 16))
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["practice5_2", "hw3_course_sample3", "hw4_course_sample3"])
def test_render_denoised_strength_zero_is_the_render(rtc, fixture):
    s = _fixture_scene(rtc, fixture)
    n = s.samples
    img, mean, st = s.RenderDenoised(0.0, seed=9)
    ref = s.Render(seed=9)
    total = s.RenderSum(seed=9, sample_count=n)
    s.close()
    assert st["passes"] == 1 and st["paths"] == n * img.shape[0] * img.shape[1]
    assert (np.abs(img.astype(int) - ref.astype(int)) <= 1).mean() >= 0.999
    want = total / np.float32(n)
    ok = np.isfinite(want) & np.isfinite(mean)
    assert ok.mean() > 0.999
    assert np.allclose(mean[ok], want[ok], rtol=1e-4, atol=1e-6)


@pytest.mark.gpu
def test_the_two_entry_points_agree(rtc):
    s = rtc.Scene(path=scene_path("practice5_1"), device=0)
    s.override(128, 96, 16)
    k = rtc.DENOISE_STRENGTH
    img, mean, _ = s.RenderDenoised(k, seed=21)
    _, halves, spp, _ = s.RenderAdaptive(0.0, min_samples=16, seed=21)
    img2, mean2 = s.Denoise(halves, spp, k)
    s.close()
    close = np.isclose(mean, mean2, rtol=1e-3, atol=1e-6) | (np.isnan(mean) & np.isnan(mean2))
    assert close.mean() >= 0.999
    assert (np.abs(img.astype(int) - img2.astype(int)) <= 1).mean() >= 0.999


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h", [("lights_mix", 96, 64), ("practice5_1", 128, 96)])
def test_denoising_lowers_the_error(rtc, name, w, h):
    s = rtc.Scene(path=scene_path(name), device=0)
    s.override(w, h, 512)
    ref = s.RenderSum(seed=977, sample_count=512).astype(np.float64) / 512
    s.override(w, h, 8)
    raw = s.RenderSum(seed=3, sample_count=8).astype(np.float64) / 8
    _, mean, _ = s.RenderDenoised(seed=3)
    s.close()
    ok = np.isfinite(ref) & np.isfinite(raw) & np.isfinite(mean)
    assert ok.mean() > 0.999
    e_raw = np.sqrt(np.mean((squash(raw[ok]) - squash(ref[ok])) ** 2))
    e_dn = np.sqrt(np.mean((squash(mean[ok]) - squash(ref[ok])) ** 2))
    m_raw, m_dn = squash(raw[ok]).mean(), squash(mean[ok]).mean()
    print("%s: rmse raw %.5f denoised %.5f (ratio %.3f), squash mean raw %.5f denoised %.5f" % (name, e_raw, e_dn, e_dn / e_raw, m_raw, m_dn))
    # measured on a B200 at k = 0.45: RMSE ratio 0.593 (lights_mix), 0.477 (practice5_1); squash means +0.21 % and +0.18 %
    # (k = 0.7 moved lights_mix's by +1.02 %: the reason the recommended strength is 0.45, DESIGN.md "Denoising")
    assert e_dn <= 0.8 * e_raw, (e_dn, e_raw)
    assert abs(m_dn - m_raw) <= 0.01 * m_raw, (m_dn, m_raw)


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw1_course_sample6", "hw2_hw2_lights"])
def test_deterministic_dialects_are_not_filtered(rtc, fixture):
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    img, mean, st = s.RenderDenoised(1.0, seed=3)
    want = s.Render(seed=3)
    frame = s.RenderSum(seed=3)
    s.close()
    assert np.array_equal(img, want)
    assert np.array_equal(mean, frame)
    assert st["passes"] == 1


@pytest.mark.gpu
def test_denoise_at_4k(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(3840, 2160, 8)
    rng = np.random.default_rng(5)
    halves = rng.uniform(0, 2, (2160, 3840, 2, 3)).astype(np.float32)
    spp = np.full((2160, 3840), 4, np.uint32)
    img, mean = s.Denoise(halves, spp, 0.5)
    s.close()
    u = (halves[:, :, 0] + halves[:, :, 1]) / np.float32(4)
    assert np.isfinite(mean).all()
    # every pixel was written by the filter: a weighted mean of its window stays within the window's range
    assert (mean >= u.min() - 1e-6).all() and (mean <= u.max() + 1e-6).all()
    assert abs(mean.mean() - u.mean()) < 0.01 and mean.std() < u.std()
    assert (np.abs(img.reshape(-1, 3)[::9973].astype(int) - to_u8(mean.reshape(-1, 3)[::9973])) <= 1).all()


@pytest.mark.gpu
def test_no_interference_with_the_other_render_paths(rtc):
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=0)
    s.override(160, 120, 8)
    before = s.RenderSum(seed=12, sample_count=8)
    want = [s.Render(seed=30 + i) for i in range(2)]
    s.RenderDenoised(seed=12)
    _, halves, spp, _ = s.RenderAdaptive(2 / 255, min_samples=2, seed=12)
    s.Denoise(halves, spp)
    after = s.RenderSum(seed=12, sample_count=8)
    ok = np.isfinite(before) & np.isfinite(after)
    assert np.allclose(before[ok], after[ok], rtol=1e-4, atol=1e-5)
    assert [np.array_equal(a, s.Render(seed=30 + i)) for i, a in enumerate(want)] == [True, True]
    got = [np.zeros_like(want[0]) for _ in range(2)]
    s.frame_begin(seed=30, slot=0)
    s.frame_begin(seed=31, slot=1)
    s.frame_end(0, got[0])
    s.frame_end(1, got[1])
    s.close()
    for a, b in zip(want, got):
        assert (np.abs(a.astype(int) - b.astype(int)) <= 1).mean() > 0.999


@pytest.mark.gpu
def test_denoise_cli(rtc, tmp_path):
    header = b"P6\n96 64\n255\n"
    outs = {}
    for name, env in (("dn", dict(RTC_DENOISE="0.45", RTC_TIMING="1")), ("zero", dict(RTC_DENOISE="0")), ("plain", {}),
                      ("adaptive", dict(RTC_DENOISE="0.45", RTC_ADAPTIVE="0.01"))):
        out = tmp_path / (name + ".ppm")
        e = dict(os.environ, RTC_SAMPLES="8", RTC_WIDTH="96", RTC_HEIGHT="64", RTC_SEED="5", **env)
        r = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path("practice5_2"), str(out)], env=e, capture_output=True, text=True)
        assert r.returncode == 0, (name, r.stderr)
        raw = out.read_bytes()
        assert raw.startswith(header) and len(raw) == len(header) + 96 * 64 * 3
        outs[name] = np.frombuffer(raw[len(header):], np.uint8).astype(int)
        if name == "dn":
            assert "passes" in r.stderr and "paths" in r.stderr
    assert (np.abs(outs["zero"] - outs["plain"]) <= 1).mean() >= 0.999
    assert (outs["dn"] != outs["plain"]).mean() > 0.1
