"""Adaptive sampling (rtc_render_adaptive / Scene.RenderAdaptive): 8x8 tiles take samples until the difference between
the means of their even and their odd samples, in display units, is below the tolerance.

The RNG is a pure function of (seed, pixel, sample, bounce), so a pixel that stopped after n samples holds the sums of
its samples [0, n): every check below compares against the oracle-pinned RenderSum, and the schedule against a numpy
restatement of the stopping rule (`model`)."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, golden, scene_path
from test_dialects import load as load_dialect

TILE = 8


# ---------------------------------------------------------------------------------------------- the rule in numpy
def aces(x):
    x = np.asarray(x, np.float32)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        num = x * (np.float32(2.51) * x + np.float32(0.03))
        den = x * (np.float32(2.43) * x + np.float32(0.59)) + np.float32(0.14)
        y = num / den
    y = np.where(y < 1, y, np.float32(1))          # std::min(1.f, y): NaN -> 1
    return np.where(y < 0, np.float32(0), y).astype(np.float32)


def display(x):
    return np.power(aces(x), np.float32(0.454545468)).astype(np.float32)


def tile_errors(A, B, n):
    """Per tile (row-major, partial at the edges) E of the half sums A, B (H, W, 3) after n samples."""
    ia, ib = np.float32(1) / np.float32((n + 1) // 2), np.float32(1) / np.float32(n // 2)
    e = np.abs(display(A * ia) - display(B * ib)).sum(2, dtype=np.float32) / np.float32(3)
    h, w = e.shape
    ty, tx = -(-h // TILE), -(-w // TILE)
    out = np.zeros((ty, tx), np.float32)
    for y in range(ty):
        for x in range(tx):
            out[y, x] = e[y * TILE:(y + 1) * TILE, x * TILE:(x + 1) * TILE].mean(dtype=np.float32)
    return out


def per_tile(a, h, w):
    """(ty, tx) tile values -> (h, w) pixel values"""
    return np.repeat(np.repeat(a, TILE, 0), TILE, 1)[:h, :w]


def model(samples, tau, min_samples, smax):
    """Replays the passes on per-sample images samples[s] (H, W, 3).  Returns the per-tile sample counts and, per tile,
    the smallest distance |E - tau| over the decisions it took part in."""
    h, w = samples.shape[1:3]
    ty, tx = -(-h // TILE), -(-w // TILE)
    n_tile = np.zeros((ty, tx), np.int64)
    margin = np.full((ty, tx), np.inf)
    active = np.ones((ty, tx), bool)
    target = min(min_samples, smax)
    while True:
        n_tile[active] = target
        if target == smax:
            break
        A = samples[0:target:2].sum(0, dtype=np.float32)
        B = samples[1:target:2].sum(0, dtype=np.float32)
        E = tile_errors(A, B, target)
        margin[active] = np.minimum(margin[active], np.abs(E[active].astype(np.float64) - tau))
        active &= ~(E < tau)
        if not active.any():
            break
        target = min(2 * target, smax)
    return n_tile, margin


def half_sums(samples, spp):
    """The model's A and B of every pixel at its own sample count"""
    A = np.zeros(samples.shape[1:], np.float32)
    B = np.zeros(samples.shape[1:], np.float32)
    for n in np.unique(spp):
        m = spp == n
        A[m] = samples[0:n:2].sum(0, dtype=np.float32)[m]
        B[m] = samples[1:n:2].sum(0, dtype=np.float32)[m]
    return A, B


def squash(x):
    return x / (1.0 + x)


# ---------------------------------------------------------------------------------------------- CPU
def test_adaptive_binding_is_declared(rtc):
    assert "rtc_render_adaptive" in rtc.exported_symbols()
    with open(rtc.HEADER_PATH) as f:
        header = f.read()
    assert "int rtc_render_adaptive(" in header and "#define RTC_ADAPTIVE_TILE 8" in header
    assert callable(rtc.load_library().rtc_render_adaptive)


@pytest.mark.parametrize("tolerance,min_samples", [(float("nan"), 16), (float("inf"), 16), (-1.0 / 255, 16), (0.01, 1), (0.01, 0)])
def test_adaptive_bad_arguments(rtc, tolerance, min_samples):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    with pytest.raises(rtc.RtcError, match="rtc error -4"):
        s.RenderAdaptive(tolerance, min_samples=min_samples)
    s.close()


def test_adaptive_host_only_scene_has_no_fallback(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    with pytest.raises(rtc.RtcError, match="rtc error -2"):
        s.RenderAdaptive(0.01, min_samples=4)
    s.close()


def test_adaptive_cli_rejects_a_bad_tolerance(rtc, tmp_path):
    for value in ("abc", "-0.5", "nan", "0.1x"):
        env = dict(os.environ, RTC_ADAPTIVE=value)
        r = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path("lights_mix"), str(tmp_path / "x.ppm")], env=env,
                           capture_output=True, text=True)
        assert r.returncode == 1, (value, r.stderr)
        assert "RTC_ADAPTIVE" in r.stderr
    env = dict(os.environ, RTC_ADAPTIVE="0.01", RTC_DEVICES="0,1")
    r = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path("lights_mix"), str(tmp_path / "x.ppm")], env=env,
                       capture_output=True, text=True)
    assert r.returncode == 1 and "one device" in r.stderr


def test_numpy_model_of_the_rule():
    """The restated rule on synthetic samples: a constant tile stops at min_samples only for tau > 0, noise keeps it."""
    rng = np.random.default_rng(3)
    smp = np.full((16, 12, 20, 3), 0.5, np.float32)
    smp[:, :, 8:16] = rng.uniform(0, 4, (16, 12, 8, 3)).astype(np.float32)   # the second tile column is noisy
    n, _ = model(smp, 0.0, 2, 16)
    assert (n == 16).all()
    n, _ = model(smp, 1e-3, 2, 16)
    assert n[0, 0] == n[1, 0] == 2 and (n[:, 1] == 16).all() and (n[:, 2] == 2).all()


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h,spp", [("lights_mix", 96, 64, 16), ("practice5_dragon_10k", 128, 128, 8)])
def test_tolerance_zero_is_the_full_render(rtc, name, w, h, spp):
    s = rtc.Scene(path=scene_path(name), device=0)
    s.override(w, h, spp)
    before = s.counters()["paths"]
    img, halves, n, st = s.RenderAdaptive(0.0, min_samples=2, seed=4)
    after = s.counters()["paths"]
    assert (n == spp).all()
    assert st["paths"] == w * h * spp == after - before
    assert st["tiles"] == math.ceil(w / 8) * math.ceil(h / 8) and st["tiles_stopped"] == 0
    assert st["passes"] == 1 + int(math.log2(spp // 2))
    want = s.RenderSum(seed=4, sample_begin=0, sample_count=spp)
    got = halves.sum(2)
    ok = np.isfinite(want) & np.isfinite(got)
    assert ok.mean() > 0.999
    assert np.allclose(got[ok], want[ok], rtol=1e-4, atol=1e-5)
    ref = s.Render(seed=4)
    assert (np.abs(img.astype(int) - ref.astype(int)) <= 1).mean() >= 0.999
    s.close()


@pytest.mark.gpu
def test_schedule_matches_the_numpy_model(rtc):
    w, h, smax, nmin, seed = 60, 44, 64, 4, 17
    s = rtc.Scene(path=scene_path("lights_mix"), device=0)
    s.override(w, h, smax)
    samples = np.stack([s.RenderSum(seed=seed, sample_begin=k, sample_count=1) for k in range(smax)])
    # a tau that leaves at least three sample counts in the model
    A, B = samples[0:nmin:2].sum(0, dtype=np.float32), samples[1:nmin:2].sum(0, dtype=np.float32)
    e0 = tile_errors(A, B, nmin)
    tau = None
    for q in (0.5, 0.4, 0.6, 0.3, 0.7, 0.2, 0.8):
        cand = float(np.float32(np.quantile(e0, q)))   # the library takes tau as a float
        if cand > 0 and len(np.unique(model(samples, cand, nmin, smax)[0])) >= 3:
            tau = cand
            break
    assert tau is not None, "no tau with three sample-count levels"
    want_n, margin = model(samples, tau, nmin, smax)
    img, halves, spp, st = s.RenderAdaptive(tau, min_samples=nmin, max_samples=smax, seed=seed)
    s.close()
    assert len(np.unique(spp)) >= 3
    got_n = spp[::TILE, ::TILE]
    clear = margin > 1e-3 * tau + 1e-6
    assert clear.mean() > 0.9
    assert np.array_equal(got_n[clear], want_n[clear]), np.argwhere(got_n != want_n)
    assert (per_tile(got_n, h, w) == spp).all()   # one count per tile
    assert st["paths"] == int(spp.sum())
    assert st["tiles_stopped"] == int((got_n < smax).sum())
    A, B = half_sums(samples, spp)
    for got, want in ((halves[:, :, 0], A), (halves[:, :, 1], B)):
        ok = np.isfinite(got) & np.isfinite(want)
        assert ok.mean() > 0.999
        assert np.allclose(got[ok], want[ok], rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_prefix_property_at_size(rtc):
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=0)
    s.override(256, 256, 64)
    for tau in (4 / 255, 2 / 255, 8 / 255, 1 / 255, 16 / 255, 0.5 / 255):
        img, halves, spp, st = s.RenderAdaptive(tau, min_samples=4, seed=23)
        if len(np.unique(spp)) >= 3:
            break
    levels = np.unique(spp)
    assert len(levels) >= 3, levels
    total = halves.sum(2)
    for n in levels:
        m = spp == n
        want = s.RenderSum(seed=23, sample_begin=0, sample_count=int(n))[m]
        ok = np.isfinite(want) & np.isfinite(total[m])
        assert ok.mean() > 0.999
        assert np.allclose(total[m][ok], want[ok], rtol=1e-4, atol=1e-5), n
    mean = total * (np.float32(1) / spp.astype(np.float32))[:, :, None]
    assert np.array_equal(img.reshape(-1, 3), s.ToUInts(mean.reshape(-1, 3)))
    s.close()


@pytest.mark.gpu
def test_statistically_matches_the_converged_reference(rtc):
    """The criterion of test_render_statistically_matches_reference, with two adaptive renders as the noise estimate."""
    smax, tau = 512, 2 / 255
    ref = golden("practice5_dragon_100k_render_96x96_512spp")["mean"].astype(np.float64)
    s = rtc.Scene(path=scene_path("practice5_dragon_100k"), device=0)
    s.override(96, 96, smax)
    est = []
    for seed in (101, 202):
        img, halves, spp, st = s.RenderAdaptive(tau, min_samples=16, max_samples=smax, seed=seed)
        est.append(halves.sum(2).astype(np.float64) / spp[:, :, None])
        # every tile that stopped early did so on its own halves
        stopped = spp[::TILE, ::TILE] < smax
        n_tile = spp[::TILE, ::TILE]
        for ty, tx in np.argwhere(stopped):
            n = int(n_tile[ty, tx])
            blk = halves[ty * TILE:(ty + 1) * TILE, tx * TILE:(tx + 1) * TILE]
            E = tile_errors(blk[:, :, 0], blk[:, :, 1], n)[0, 0]
            assert E < tau * (1 + 1e-3) + 1e-6, (ty, tx, n, E)
        assert st["tiles_stopped"] == int(stopped.sum())
    s.close()
    a, b = est
    ok = np.isfinite(ref) & np.isfinite(a) & np.isfinite(b)
    assert ok.mean() > 0.999
    sa, sb, sr = squash(a[ok]), squash(b[ok]), squash(ref[ok])
    noise = np.sqrt(np.mean((sa - sb) ** 2))
    err = np.sqrt(np.mean((sa - sr) ** 2))
    assert err <= 1.2 * noise + 1e-4, (err, noise)
    diff = sa - sr
    se = diff.std() / np.sqrt(diff.size) + 1e-12
    assert abs(diff.mean()) < 4 * se + 2e-4, (diff.mean(), se)


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw3_course_sample3", "hw4_course_sample3"])
def test_monte_carlo_dialects_at_tolerance_zero(rtc, fixture):
    """The list generator keeps hw3's half-pixel jitter offset: tau = 0 is RenderSum in every dialect."""
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    spp = min(s.samples, 16)
    s.override(-1, -1, spp)
    img, halves, n, st = s.RenderAdaptive(0.0, min_samples=2, seed=8)
    want = s.RenderSum(seed=8, sample_begin=0, sample_count=spp)
    s.close()
    assert (n == spp).all()
    got = halves.sum(2)
    ok = np.isfinite(want) & np.isfinite(got)
    assert ok.mean() > 0.999
    assert np.allclose(got[ok], want[ok], rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["hw1_course_sample6", "hw2_hw2_lights"])
def test_deterministic_dialects_render_their_one_frame(rtc, fixture):
    text, dialect, _ = load_dialect(fixture)
    s = rtc.Scene(text=text, device=0, dialect=dialect)
    img, halves, n, st = s.RenderAdaptive(0.01, min_samples=4, seed=3)
    want = s.Render(seed=3)
    frame = s.RenderSum(seed=3)
    s.close()
    assert (n == 1).all()
    assert np.array_equal(img, want)
    assert np.array_equal(halves[:, :, 0], frame) and not halves[:, :, 1].any()
    assert st["passes"] == 1 and st["tiles_stopped"] == 0


def _run_cli(tmp_path, name, **env):
    out = tmp_path / name
    e = dict(os.environ, RTC_SAMPLES="8", RTC_WIDTH="96", RTC_HEIGHT="64", RTC_SEED="5", **env)
    r = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path("practice5_2"), str(out)], env=e, capture_output=True, text=True)
    return r, out


@pytest.mark.gpu
def test_adaptive_cli(rtc, tmp_path):
    header = b"P6\n96 64\n255\n"
    r, out = _run_cli(tmp_path, "a.ppm", RTC_ADAPTIVE="0.01", RTC_TIMING="1")
    assert r.returncode == 0, r.stderr
    raw = out.read_bytes()
    assert raw.startswith(header) and len(raw) == len(header) + 96 * 64 * 3
    assert "adaptive:" in r.stderr and "passes" in r.stderr and "paths" in r.stderr
    r, zero = _run_cli(tmp_path, "zero.ppm", RTC_ADAPTIVE="0")
    assert r.returncode == 0, r.stderr
    r, plain = _run_cli(tmp_path, "plain.ppm")
    assert r.returncode == 0, r.stderr
    a = np.frombuffer(zero.read_bytes()[len(header):], np.uint8).astype(int)
    b = np.frombuffer(plain.read_bytes()[len(header):], np.uint8).astype(int)
    assert a.size == b.size == 96 * 64 * 3
    assert (np.abs(a - b) <= 1).mean() >= 0.999
    r, _ = _run_cli(tmp_path, "bad.ppm", RTC_ADAPTIVE="abc")
    assert r.returncode == 1


@pytest.mark.gpu
def test_no_interference_with_the_other_render_paths(rtc):
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=0)
    s.override(160, 120, 8)
    before = s.RenderSum(seed=12, sample_count=8)
    want = [s.Render(seed=30 + i) for i in range(2)]
    s.RenderAdaptive(2 / 255, min_samples=2, seed=12)
    after = s.RenderSum(seed=12, sample_count=8)
    ok = np.isfinite(before) & np.isfinite(after)
    assert np.allclose(before[ok], after[ok], rtol=1e-4, atol=1e-5)
    got = [np.zeros_like(want[0]) for _ in range(2)]
    s.frame_begin(seed=30, slot=0)
    s.frame_begin(seed=31, slot=1)
    s.frame_end(0, got[0])
    s.frame_end(1, got[1])
    s.close()
    for a, b in zip(want, got):
        assert (np.abs(a.astype(int) - b.astype(int)) <= 1).mean() > 0.999
