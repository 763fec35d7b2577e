"""The thin-lens camera (rtc_scene_set_lens, DESIGN.md "Thin lens").

CPU: the host-side state and its checks; the depth of field the lens makes in the oracle's render
(tests/host_emul/lens_oracle.c) against the thin-lens blur radius.
GPU: every render path through the lens against the oracle and against each other; lens renders build no camera lists."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import orclib
from conftest import ROOT, golden, scene_path
from test_camera_lists import TRAVERSE
from test_views import orbit, raw_lib, render_close, text_of, u8_close

EMU_DIR = os.path.join(ROOT, "tests", "host_emul")
RTC_ERR_ARG, RTC_ERR_UNSUPPORTED = -4, -5
f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


def stale(so, srcs):
    return not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(p) for p in srcs)


@pytest.fixture(scope="module")
def lens_oracle():
    """orc_render_sum_lens: the oracle's render with the lens step in its camera sample."""
    so = os.path.join(EMU_DIR, "liblens_oracle.so")
    srcs = [os.path.join(EMU_DIR, "lens_oracle.c"), os.path.join(ROOT, "oracle", "rt_oracle.c")]
    if stale(so, srcs):
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                               srcs[0], "-o", so, "-lm"])
    L = C.CDLL(so)
    L.orc_scene_parse_dialect.restype = C.c_void_p
    L.orc_scene_parse_dialect.argtypes = [C.c_char_p, C.c_long, C.c_int]
    L.orc_scene_free.argtypes = [C.c_void_p]
    L.orc_scene_override.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.orc_render_sum.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_long, C.c_long, f32p, u64p, C.c_int]
    L.orc_render_sum_lens.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_uint32, C.c_uint32, C.c_uint32, C.c_long, C.c_long,
                                      f32p, u64p, C.c_int]
    return L


def lens_render(L, text, r, f, seed, sample_begin, spp, w, h, dialect=5, lens=True, depth=-1):
    """(sums (w h, 3), paths, rays) of the oracle with a lens (lens=False: orc_render_sum itself)"""
    b = text.encode()
    s = L.orc_scene_parse_dialect(b, len(b), dialect)
    assert s
    try:
        L.orc_scene_override(s, w, h, spp, depth)
        out = np.zeros((w * h, 3), np.float32)
        cnt = np.zeros(2, np.uint64)
        if lens:
            L.orc_render_sum_lens(s, r, f, seed, sample_begin, spp, 0, w * h, out, cnt, 0)
        else:
            L.orc_render_sum(s, seed, sample_begin, spp, 0, w * h, out, cnt, 0)
        return out, int(cnt[0]), int(cnt[1])
    finally:
        L.orc_scene_free(s)


def focus_and_scale(text, dialect):
    """(f, world units per pixel of blur per unit r / f): f = the median forward distance of the primary hits of a grid of
    pixel-centre rays (t is the forward distance: d's forward coefficient is 1), the blur radius of a point at depth z
    being r |z - f| / z * W / (2 f tan(fov_x / 2)) pixels."""
    a = orclib.Scene(orclib.oracle(), text=text, dialect=dialect)
    try:
        o, d = orclib.pixel_center_rays(a, step=max(1, a.width // 24))
        pid, t, _, _ = a.intersect(o, d)
        cam = a.camera()
        f = float(np.median(t[pid >= 0])) if (pid >= 0).any() else 1.0
        return f, a.width, math.tan(float(cam[12]) / 2)
    finally:
        a.close()


def aperture_for_blur(f, width, tan_half, pixels):
    """r whose blur of the far background (z -> inf: r |z - f| / z -> r) is `pixels` pixels in radius"""
    return pixels * 2 * f * tan_half / width


# ---------------------------------------------------------------------------------------------------- CPU: host state
def test_lens_round_trip_and_set_camera_keeps_it(rtc):
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    assert s.lens() == (0.0, 1.0)
    s.set_lens(0.125, 6.5)
    assert s.lens() == (0.125, 6.5)
    s.set_camera(orbit(s.camera(), 0.3))
    assert s.lens() == (0.125, 6.5)
    s.set_lens(0.0, 2.0)
    assert s.lens() == (0.0, 2.0)
    s.close()


def test_bad_lenses_are_refused_before_any_change(rtc):
    lib = raw_lib(rtc)
    lib.rtc_scene_set_lens.argtypes = [C.c_void_p, C.c_float, C.c_float]
    lib.rtc_scene_set_lens.restype = C.c_int
    lib.rtc_scene_lens.argtypes = [C.c_void_p, C.c_void_p]
    lib.rtc_scene_lens.restype = C.c_int
    assert lib.rtc_scene_set_lens(None, 0.1, 1.0) == RTC_ERR_ARG
    out = np.zeros(2, np.float32)
    assert lib.rtc_scene_lens(None, out.ctypes.data_as(C.c_void_p)) == RTC_ERR_ARG
    s = rtc.Scene(path=scene_path("lights_mix"), device=-1)
    s.set_lens(0.25, 4.0)
    bad = [(float("nan"), 1.0), (0.1, float("nan")), (float("inf"), 1.0), (-float("inf"), 1.0), (0.1, float("inf")),
           (0.1, -float("inf")), (-0.01, 1.0), (0.1, 0.0), (0.1, -2.0), (0.0, 0.0)]
    for r, f in bad:
        assert lib.rtc_scene_set_lens(C.c_void_p(s.h), r, f) == RTC_ERR_ARG, (r, f)
        assert s.lens() == (0.25, 4.0)
    s.close()


@pytest.mark.parametrize("fixture", ["hw1_course_sample6", "hw2_hw2_lights"])
def test_deterministic_dialects_refuse_an_aperture(rtc, fixture):
    g = golden(fixture)
    s = rtc.Scene(text=bytes(g["text"]).decode(), device=-1, dialect=int(g["dialect"]))
    with pytest.raises(RuntimeError) as e:
        s.set_lens(0.1, 3.0)
    assert str(RTC_ERR_UNSUPPORTED) in str(e.value)
    assert s.lens() == (0.0, 1.0)
    s.set_lens(0.0, 3.0)   # the pinhole with another focus distance is still the pinhole
    assert s.lens() == (0.0, 3.0)
    s.close()


def test_header_and_signatures(rtc):
    header = open(os.path.join(ROOT, "include", "rtc_b200.h")).read()
    assert "int rtc_scene_set_lens(rtc_scene* s, float aperture_radius, float focus_distance);" in header
    assert "int rtc_scene_lens(const rtc_scene* s, float out[2]);" in header
    assert {"rtc_scene_set_lens", "rtc_scene_lens"} <= set(rtc.exported_symbols())


# ---------------------------------------------------------------------------------------------------- CPU: oracle physics
# Two emissive slabs facing the camera, each with a vertical edge on the image's centre column: one at depth Z1 (in
# focus) in the upper rows, one at Z2 in the lower rows; RAY_DEPTH 1, so a sample is 1 where it hits a slab, else 0.
W, H, Z1, Z2 = 96, 48, 4.0, 8.0
TWO_BOXES = """DIMENSIONS %d %d
RAY_DEPTH 1
SAMPLES 1
BG_COLOR 0 0 0
CAMERA_POSITION 0 0 0
CAMERA_RIGHT 1 0 0
CAMERA_UP 0 1 0
CAMERA_FORWARD 0 0 1
CAMERA_FOV_X %.9g

NEW_PRIMITIVE
BOX 10 1.4 0.01
POSITION -10 1.6 %g
EMISSION 1 1 1

NEW_PRIMITIVE
BOX 10 2 0.01
POSITION -10 -2.4 %g
EMISSION 1 1 1
""" % (W, H, 2 * math.atan(0.5), Z1, Z2)


def edge_width(sums, spp, rows):
    """10-90 % width in pixels of the edge (1 on the left, 0 on the right) of the mean over `rows`"""
    p = sums.reshape(H, W, 3)[rows, :, 0].mean(0) / spp
    def cross(level):
        i = int(np.nonzero(p < level)[0][0])
        return i - 1 + (p[i - 1] - level) / (p[i - 1] - p[i]) + 0.5
    return cross(0.1) - cross(0.9)


def model_edge_width(radius):
    """10-90 % width of the edge of a uniform disk of `radius` pixels convolved with the 1-pixel jitter box"""
    xs = np.linspace(-radius - 2, radius + 2, 4001)
    h = np.clip(xs[:, None] - np.linspace(-0.5, 0.5, 201)[None, :], -radius, radius) / max(radius, 1e-9)
    seg = (np.arccos(h) - h * np.sqrt(1 - h * h)) / math.pi   # share of the disk beyond the line at h radii
    esf = seg.mean(1)[::-1]   # falling in x: reversed for np.interp
    return float(np.interp(0.1, esf, xs[::-1]) - np.interp(0.9, esf, xs[::-1]))


def test_oracle_depth_of_field_matches_the_thin_lens(lens_oracle):
    spp, f = 512, Z1
    pin, _, _ = lens_render(lens_oracle, TWO_BOXES, 0.0, f, 5, 0, spp, W, H)
    top, bottom = slice(5, 12), slice(34, 43)
    for r in (0.2, 0.5):
        got, paths, _ = lens_render(lens_oracle, TWO_BOXES, r, f, 5, 0, spp, W, H)
        assert paths == W * H * spp
        radius = r * abs(Z2 - f) / Z2 * W / (2 * f * 0.5)   # the far slab's blur radius in pixels
        want = model_edge_width(radius)
        measured = edge_width(got, spp, bottom)
        print("r %.2f: blur radius %.2f px, edge width %.2f px (disk model %.2f, pinhole %.2f)"
              % (r, radius, measured, want, edge_width(pin, spp, bottom)))
        assert abs(measured - want) <= 0.25 * want
        assert abs(edge_width(got, spp, top) - edge_width(pin, spp, top)) < 1.0


def test_oracle_lens_radius_zero_is_the_pinhole(lens_oracle):
    text = text_of("lights_mix")
    a, pa, ra = lens_render(lens_oracle, text, 0.0, 3.0, 7, 1, 4, 48, 32)
    b, pb, rb = lens_render(lens_oracle, text, 0.0, 3.0, 7, 1, 4, 48, 32, lens=False)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and (pa, ra) == (pb, rb)


# ---------------------------------------------------------------------------------------------------- GPU
def focused(rtc, name):
    """(scene on device 0, f, tan(fov_x / 2)): the scene focused on the subject, the forward distance of the primary hit
    of the centre pixel, or the median over a grid when the centre ray misses"""
    s = rtc.Scene(path=scene_path(name), device=0)
    f, _, tan_half = focus_and_scale(text_of(name), 5)
    return s, f, tan_half


def good_share(got, want):
    """render_close's per-pixel criterion: the share of pixels within 2e-3 relative"""
    ok = np.isfinite(want).all(1) & np.isfinite(got).all(1)
    rel = np.abs(got - want).max(1) / (np.abs(want).max(1) + 1e-3)
    return float(((rel <= 2e-3) & ok).mean())


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h,spp,depth", [("lights_mix", 48, 32, 64, 1), ("practice5_dragon_10k", 64, 64, 32, -1),
                                                ("practice5_dragon_100k", 48, 48, 16, -1)])
def test_lens_render_sample_exact_vs_oracle(rtc, lens_oracle, name, w, h, spp, depth):
    """The same Philox streams through the same lens on both sides.  lights_mix at RAY_DEPTH 1: its camera rays and their
    first hits (its deeper bounces differ from the oracle's in a few percent of pixels at this spp with or without a
    lens: test_lens_lights_mix_full_depth_as_close_as_the_pinhole)."""
    s, f, tan_half = focused(rtc, name)
    s.override(w, h, spp, depth)
    for blur in (3, 30):
        r = aperture_for_blur(f, w, tan_half, blur)
        s.set_lens(r, f)
        s.reset_counters()
        got = s.RenderSum(seed=9, sample_begin=2, sample_count=spp).reshape(-1, 3)
        cnt = s.counters()
        want, paths, rays = lens_render(lens_oracle, text_of(name), np.float32(r), np.float32(f), 9, 2, spp, w, h, depth=depth)
        assert cnt["paths"] == paths == w * h * spp
        assert abs(cnt["rays"] - rays) <= 1e-3 * rays
        render_close(got, want)
    s.close()


@pytest.mark.gpu
def test_lens_lights_mix_full_depth_as_close_as_the_pinhole(rtc, lens_oracle):
    """lights_mix at full depth and 64 spp: the pinhole itself agrees with the oracle in 98.4 % of pixels (later bounces
    through its ellipsoid light and glossy surfaces), below render_close's 99 %.  Through the lens, the share stays within
    a percent of the pinhole's, and the medians agree."""
    name, w, h, spp = "lights_mix", 48, 32, 64
    s, f, tan_half = focused(rtc, name)
    s.override(w, h, spp)
    pin = good_share(s.RenderSum(seed=9, sample_begin=2, sample_count=spp).reshape(-1, 3),
                     lens_render(lens_oracle, text_of(name), 0.0, np.float32(f), 9, 2, spp, w, h)[0])
    for blur in (3, 30):
        r = aperture_for_blur(f, w, tan_half, blur)
        s.set_lens(r, f)
        got = s.RenderSum(seed=9, sample_begin=2, sample_count=spp).reshape(-1, 3)
        want, _, _ = lens_render(lens_oracle, text_of(name), np.float32(r), np.float32(f), 9, 2, spp, w, h)
        share = good_share(got, want)
        print("lights_mix blur %d: %.4f of pixels within 2e-3 (pinhole %.4f)" % (blur, share, pin))
        assert share >= pin - 0.01
        sq = lambda x: x / (1.0 + x)   # noqa: E731
        assert abs(np.median(sq(got)) - np.median(sq(want))) < 1e-3
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lights_mix", "practice5_dragon_100k"])
def test_lens_renders_build_no_lists(rtc, name):
    """With a lens every camera ray takes the index traversal (DESIGN.md "Thin lens": the lists of lens beams were
    slower): RenderSum equals RenderViews of the scene's own camera, which never builds lists, and no ray is listed."""
    s, f, tan_half = focused(rtc, name)
    s.override(64, 64, 8)
    for blur in (3, 30):
        s.set_lens(aperture_for_blur(f, 64, tan_half, blur), f)
        s.reset_counters()
        got = s.RenderSum(seed=4, sample_begin=0, sample_count=8)
        assert s.camera_list_rays() == 0
        assert (s.camera_list_lengths() == TRAVERSE).all()
        _, views = s.RenderViews([s.camera()], seed=4, want_sum=True)
        assert np.allclose(got, views[0], rtol=1e-4, atol=1e-5), np.abs(got - views[0]).max()
    s.set_lens(0.0, f)   # back to the pinhole: its camera rays come from lists again
    s.reset_counters()
    s.RenderSum(seed=4, sample_begin=0, sample_count=8)
    assert s.camera_list_rays() > 0
    s.close()


@pytest.mark.gpu
def test_every_render_path_takes_the_lens(rtc):
    import torch  # noqa: F401  (RenderMulti's peer path wants the CUDA context of torch's process set up alike)
    name, w, h, spp = "lights_mix", 48, 40, 8
    s, f, tan_half = focused(rtc, name)
    s.override(w, h, spp)
    s.set_lens(aperture_for_blur(f, w, tan_half, 6), f)
    ref = s.RenderSum(seed=2, sample_begin=0, sample_count=spp)
    pin = rtc.Scene(path=scene_path(name), device=0)
    pin.override(w, h, spp)
    assert not np.allclose(ref, pin.RenderSum(seed=2, sample_begin=0, sample_count=spp), rtol=1e-3)   # the lens matters
    img, sm = s.RenderMulti([0, 0], seed=2, want_sum=True)
    assert np.allclose(sm, ref, rtol=1e-4, atol=1e-5)
    u8_close(img, s.Render(seed=2))
    # adaptive at tolerance 0: every pixel at SAMPLES; the half sums are the even and the odd samples
    single = [s.RenderSum(seed=2, sample_begin=k, sample_count=1) for k in range(spp)]
    even, odd = sum(single[0::2]), sum(single[1::2])
    for _, halves, px, _ in (s.RenderAdaptive(0.0, min_samples=4, seed=2), s.RenderAdaptiveMulti([0, 0], 0.0, min_samples=4, seed=2)):
        assert (px == spp).all()
        assert np.allclose(halves[:, :, 0], even, rtol=1e-4, atol=1e-5)
        assert np.allclose(halves[:, :, 1], odd, rtol=1e-4, atol=1e-5)
    _, mean, _ = s.RenderDenoised(strength=0.0, seed=2)
    assert np.allclose(mean, ref / spp, rtol=1e-3, atol=1e-4)
    frame = np.zeros((h, w, 3), np.uint8)
    s.frame_begin(seed=2, slot=0)
    s.frame_end(0, frame)
    u8_close(frame, s.Render(seed=2))
    # the views of an orbit, each through the lens with its own axes
    base = s.camera()
    cams = np.stack([orbit(base, a) for a in (-0.3, 0.0, 0.25)])
    _, sums = s.RenderViews(cams, seed=2, want_sum=True)
    for v in range(len(cams)):
        s.set_camera(cams[v])
        assert np.allclose(sums[v], s.RenderSum(seed=2, sample_begin=0, sample_count=spp), rtol=1e-4, atol=1e-5), v
    s.set_camera(base)
    pin.close()
    s.close()


@pytest.mark.gpu
def test_back_to_the_pinhole(rtc):
    name = "practice5_dragon_10k"
    s, f, _ = focused(rtc, name)
    s.override(64, 64, 4)
    s.set_lens(0.3, f)
    s.RenderSum(seed=1, sample_begin=0, sample_count=4)
    s.set_lens(0.0, f)
    fresh = rtc.Scene(path=scene_path(name), device=0)
    fresh.override(64, 64, 4)
    assert np.allclose(s.RenderSum(seed=1, sample_begin=0, sample_count=4), fresh.RenderSum(seed=1, sample_begin=0, sample_count=4),
                       rtol=1e-4, atol=1e-5)
    u8_close(s.Render(seed=1), fresh.Render(seed=1))
    s.close()
    fresh.close()


@pytest.mark.gpu
def test_far_lens_rebuilds_the_index_tree(rtc, oracle_lib, lens_oracle):
    """A lens whose origins reach 40x the extent the index BVH was built for: the tree is rebuilt and uploaded again
    (arena_check, the replica of RenderMulti), and rays from such origins hit what the oracle's reference tree hits."""
    name = "practice5_dragon_100k"
    s, f, _ = focused(rtc, name)
    s.override(32, 32, 2)
    s.RenderMulti([0, 0])   # the replica, with the tree built at load
    cam = s.camera()
    r = 40 * 15.0
    s.set_lens(r, f)
    assert s.arena_check() == 0
    rng = np.random.default_rng(3)
    n = 4096
    ang, rad = rng.random(n) * 2 * np.pi, np.sqrt(rng.random(n))
    e = (rad * np.cos(ang))[:, None] * cam[3:6][None] + (rad * np.sin(ang))[:, None] * cam[6:9][None]
    pos, fwd = cam[0:3].astype(np.float64), cam[9:12].astype(np.float64)
    target = pos + f * fwd + (rng.random((n, 2)) - 0.5) @ np.stack([cam[3:6], cam[6:9]]) * 0.3 * f
    o = (pos + r * e).astype(np.float32)
    d = (target - o).astype(np.float32)
    pid, t, _, _ = s.RayIntersection(o, d, rtc.TRAVERSAL_INDEX)
    a = orclib.Scene(oracle_lib, scene_path(name))
    wpid, wt, _, _ = a.intersect(o, d)
    a.close()
    assert (wpid >= 0).mean() > 0.2
    assert (pid == wpid).mean() >= 0.9999, int((pid != wpid).sum())
    img, sm = s.RenderMulti([0, 0], seed=4, want_sum=True)
    one = s.RenderSum(seed=4, sample_begin=0, sample_count=2)
    assert np.allclose(sm, one, rtol=1e-4, atol=1e-5)
    want, _, _ = lens_render(lens_oracle, text_of(name), np.float32(r), np.float32(f), 4, 0, 2, 32, 32)
    render_close(one.reshape(-1, 3), want)
    s.close()


@pytest.mark.gpu
def test_rtc_lens_cli(rtc, tmp_path):
    name = "lights_mix"
    s, f, tan_half = focused(rtc, name)
    r = aperture_for_blur(f, s.width, tan_half, 5)
    s.set_lens(np.float32(r), np.float32(f))
    want = s.Render(seed=0)
    s.close()
    env = dict(os.environ, RTC_LENS="%.9g,%.9g" % (np.float32(r), np.float32(f)))
    out = tmp_path / "lens.ppm"
    subprocess.check_call([os.path.join(ROOT, "run.sh"), scene_path(name), str(out)], env=env)
    u8_close(orclib.read_ppm(str(out)), want)
    for value in ("0.1", "0.1,", ",2", "a,b", "0.1,2,3", "-0.1,2", "0.1,0", "nan,1"):
        env = dict(os.environ, RTC_LENS=value)
        p = subprocess.run([os.path.join(ROOT, "run.sh"), scene_path(name), str(tmp_path / "x.ppm")], env=env,
                           capture_output=True, text=True)
        assert p.returncode == 1 and "RTC_LENS" in p.stderr, (value, p.returncode, p.stderr)
