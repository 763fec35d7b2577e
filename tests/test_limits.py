"""Scenes at the library's limits (DESIGN.md "Limits") and past the capacity of the index traversal, against the oracle.

* Fallback.  A ray whose index traversal records more than kMaxRecords = 24 reference leaves with a hit walks the
  reference tree instead (`trace_reftree`): in k_traverse (renders and RayIntersection) and in `collect_leaf_hits`
  (the hw1 / hw2 kernels).  No shipped scene has such rays.  A "fence" of thin boxes along the view axis and a stack of
  triangles on parallel planes have them from 25 primitives on.  With a plane between the stack's rendered triangles
  and their boxes, the answer also depends on the walk starting from the plane's distance.  The other trigger, a full
  traversal stack, is not reached by any scene here.
* Accepted edges: a reference leaf of 64 primitives, RAY_DEPTH 62 (the last of the 64 per-bounce queue slots) and hw2
  at RAY_DEPTH 32 (the Whitted stack of 34 entries).  One more is refused.
* Boxes whose surface areas reach the SAH's 1e18 "infinity" leave the reference's builder without a cut; the library
  refuses such a scene instead of recursing until the stack overflows.

The GPU tests that render these scenes against the oracle with the common tolerances are the `fence_25`,
`triangle_stack_25` and `closed_room_depth_62` inputs of test_gpu_parity.py `test_edge_scenes_vs_oracle`."""
import subprocess
import sys

import numpy as np
import pytest

import orclib
from conftest import ROOT
from test_host_emulation import emu, emu_intersect  # noqa: F401  (emu is a fixture)

K_MAX_RECORDS = 24

HEAD = ("DIMENSIONS 64 48\nSAMPLES 4\nRAY_DEPTH 6\nBG_COLOR 0.2 0.3 0.4\nCAMERA_POSITION 0 0 0\nCAMERA_RIGHT 1 0 0\n"
        "CAMERA_UP 0 1 0\nCAMERA_FORWARD 0 0 -1\nCAMERA_FOV_X 1.0\n")


def fence(n):
    """n thin boxes 0.5 apart along the view axis (each its own reference leaf: a ray along the axis records n leaves)
    and a tilted plane in the gap behind the 13th box.  Every box has a colour of its own, so that an hw1 frame shows
    which one was hit.  The text reads as hw1 as well as hw5."""
    boxes = "".join("NEW_PRIMITIVE\nBOX 0.6 0.6 0.05\nPOSITION 0 0 %g\nCOLOR %.4f 0.5 0.5\n\n" % (-2 - 0.5 * i, (i + 1) / (n + 1))
                    for i in range(n))
    return HEAD + boxes + "NEW_PRIMITIVE\nPLANE 0.3 0 1\nPOSITION 0 0 -8.2\nCOLOR 0.3 0.7 0.3\n"


def triangle_stack(n, plane=False):
    """n equal triangles on parallel planes 0.1 apart.  A triangle is rendered on the parallel plane through the origin
    (DESIGN.md "Traversal", fact 1), so the hits of a ray on all n tie in t and the reference's tree order decides.

    With `plane`, a plane lies between the rendered triangles (z = 0) and their boxes (z = -2 and beyond).  The reference
    walk starts with the plane's distance as its closest hit and skips every box that lies behind it, so a ray that
    meets a triangle in front of the plane still ends on the plane: only a walk that starts from the plane's distance,
    as the one that replaces the index traversal must, gives the reference's answer."""
    tris = "".join("NEW_PRIMITIVE\nTRIANGLE -1 -1 %g 1 -1 %g 0 1 %g\nCOLOR 0.5 0.5 0.5\n\n" % ((-2 - 0.1 * i,) * 3)
                   for i in range(n))
    wall = "NEW_PRIMITIVE\nPLANE 0 0 1\nPOSITION 0 0 -1\nCOLOR 0.3 0.6 0.3\n" if plane else ""
    return HEAD.replace("CAMERA_POSITION 0 0 0", "CAMERA_POSITION 0 0 5") + tris + wall


FALLBACK_SCENES = {"fence_24": (fence(24), 24), "fence_25": (fence(25), 25), "fence_40": (fence(40), 40),
                   "triangle_stack_24": (triangle_stack(24), 24), "triangle_stack_25": (triangle_stack(25), 25),
                   "triangle_stack_plane_25": (triangle_stack(25, plane=True), 25)}


def fence_rays(scene, seed=1, n=20000):
    """Every pixel centre, and rays close to the view axis in either direction from origins in front of, inside and
    behind the fence: they pass through many boxes, and the first one they hit varies with the origin."""
    o, d = orclib.pixel_center_rays(scene)
    rng = np.random.default_rng(seed)
    o2 = np.stack([rng.normal(0, 0.3, n), rng.normal(0, 0.3, n), rng.uniform(-22, 6, n)], 1)
    d2 = np.stack([rng.normal(0, 0.05, n), rng.normal(0, 0.05, n), np.where(rng.uniform(size=n) < 0.7, -1.0, 1.0)], 1)
    d2 /= np.linalg.norm(d2, axis=1, keepdims=True)
    return np.concatenate([o, o2.astype(np.float32)]), np.concatenate([d, d2.astype(np.float32)])


def same(a, b):
    """Equal values (a zero component of a normal may differ in sign)."""
    return a.shape == b.shape and np.array_equal(a, b)


def parsed(L, text, dialect=5):
    raw = text.encode()
    h = L.emu_scene_parse_dialect(raw, len(raw), dialect)
    assert h
    return h


# --------------------------------------------------------------------------------------- CPU: host emulation, fallback
@pytest.mark.parametrize("name", sorted(FALLBACK_SCENES))
def test_fallback_boundary_in_host_emulation(emu, oracle_lib, name):
    """The device code compiled for the host: id, t, normal and interior equal to the oracle's, in both traversal
    modes.  The index traversal gives up on exactly the rays that record a 25th leaf: none at 24 primitives, some
    at 25."""
    text, nprims = FALLBACK_SCENES[name]
    a = orclib.Scene(oracle_lib, text=text)
    o, d = fence_rays(a)
    want = a.intersect(o, d)
    a.close()
    assert len(np.unique(want[0])) > (10 if name.startswith("fence") else 1)   # the rays do not all end on one primitive
    h = parsed(emu, text)
    for mode in (0, 1):
        *got, st = emu_intersect(emu, h, o, d, mode)
        for g, w, what in zip(got, want, ("id", "t", "normal", "interior")):
            assert same(g, w), (name, mode, what, int((g != w).reshape(len(o), -1).any(1).sum()))
        if mode == 0:
            fallbacks = int(st[1])
    emu.emu_scene_free(h)
    if nprims <= K_MAX_RECORDS:
        assert fallbacks == 0, fallbacks
    else:
        assert fallbacks > 0


def test_hw1_fence_in_host_emulation(emu, oracle_lib):
    """hw1 ray casting (`collect_leaf_hits` and its fallback) on the 40-box fence: the frame is exactly the oracle's,
    and its pixel-centre rays do fall back."""
    text = fence(40)
    a = orclib.Scene(oracle_lib, text=text, dialect=1)
    want = a.render_sum(0, 0, 1)[0]
    o, d = orclib.pixel_center_rays(a)
    a.close()
    h = parsed(emu, text, dialect=1)
    lin = np.zeros(want.shape, np.float32)
    assert emu.emu_frame_linear(h, lin) == 0
    assert same(lin, want)
    assert emu_intersect(emu, h, o, d, 0)[4][1] > 0
    emu.emu_scene_free(h)


# ------------------------------------------------------------------------------- CPU: a reference leaf of 64 primitives
# With every POSITION at the origin all sort keys are equal, and libstdc++'s std::sort of 64 (and of 65) such entries
# puts these file positions first and last on each of the builder's three axis sorts.  The SAH keeps a leaf when every
# cut has a box as large as the whole leaf on both sides; the ellipsoids there are unit spheres, so it keeps them all.
LEAF_ANCHORS = (0, 7, 30, 31, 40, 42, 48, 63)


def ellipsoid_leaf(n):
    """n overlapping ellipsoids about the origin, all in one reference leaf, with the camera inside them.  Apart from
    the unit spheres of LEAF_ANCHORS their radii lie between 0.75 and 1 and differ per axis, so that which one a ray
    meets first depends on its origin and direction rather than on the order in which ties are broken."""
    rng = np.random.default_rng(3)
    head = HEAD.replace("CAMERA_POSITION 0 0 0", "CAMERA_POSITION 0.05 0.1 0.2").replace("CAMERA_FOV_X 1.0", "CAMERA_FOV_X 2.0")
    out = [head]
    for i in range(n):
        r = (1.0, 1.0, 1.0) if i in LEAF_ANCHORS else tuple(1 - 0.25 * rng.uniform(size=3))
        out.append("NEW_PRIMITIVE\nELLIPSOID %.6g %.6g %.6g\nCOLOR 0.5 0.5 0.5\n\n" % r)
    return "".join(out)


def leaf_rays(scene, seed=2, n=20000):
    o, d = orclib.pixel_center_rays(scene)
    rng = np.random.default_rng(seed)
    o2 = rng.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    d2 = rng.normal(size=(n, 3)).astype(np.float32)
    return np.concatenate([o, o2]), np.concatenate([d, d2])


def test_leaf_of_64_primitives_vs_oracle(rtc, emu, oracle_lib):
    """The largest leaf the library accepts: one leaf of 64 in the host tree, node for node the oracle's, and the device
    code's hits exactly the oracle's.  65 primitives in one leaf are refused."""
    text = ellipsoid_leaf(64)
    s = rtc.Scene(text=text, device=-1)
    a = orclib.Scene(oracle_lib, text=text)
    aabb, links, root = s.nodes()
    assert s.nnodes == 1 and links[root].tolist() == [0xFFFFFFFF, 0xFFFFFFFF, 0, 64]
    oaabb, olinks, oroot = a.nodes()
    assert np.array_equal(aabb.view(np.uint32), oaabb.view(np.uint32)) and np.array_equal(links, olinks) and root == oroot
    assert np.array_equal(s.prim_order(), a.prim_order())
    s.close()
    o, d = leaf_rays(a)
    want = a.intersect(o, d)
    a.close()
    assert len(np.unique(want[0])) > 40
    h = parsed(emu, text)
    for mode in (0, 1):
        got = emu_intersect(emu, h, o, d, mode)[:4]
        for g, w, what in zip(got, want, ("id", "t", "normal", "interior")):
            assert same(g, w), (mode, what)
    emu.emu_scene_free(h)
    with pytest.raises(rtc.RtcError, match="more than 64 primitives"):
        rtc.Scene(text=ellipsoid_leaf(65), device=-1)


# ------------------------------------------------------------------------------------------ CPU: the deepest paths
# A closed room: the camera inside a large diffuse BOX and a small emitter that reflects (METALLIC), so that no path
# leaves the room and none ends on the emitter.  Nearly every path takes all RAY_DEPTH bounces.
CLOSED_ROOM = """DIMENSIONS 32 24
SAMPLES 4
RAY_DEPTH 62
BG_COLOR 1 0 1
CAMERA_POSITION 0 0 2
CAMERA_RIGHT 1 0 0
CAMERA_UP 0 1 0
CAMERA_FORWARD 0 0 -1
CAMERA_FOV_X 1.2

NEW_PRIMITIVE
BOX 3 2 4
COLOR 0.8 0.75 0.7

NEW_PRIMITIVE
ELLIPSOID 0.3 0.1 0.3
POSITION 0 1.85 -1
EMISSION 20 18 15
METALLIC
COLOR 0.5 0.5 0.5
"""

# hw2 at its deepest: a ray that enters the glass ball is reflected inside it at every hit, and each hit also sends a
# refracted ray out, so the Whitted recursion runs the full RAY_DEPTH with one more pending ray per level.
WHITTED_DEEPEST = """RAY_DEPTH 32
DIMENSIONS 64 48
BG_COLOR 0.35 0.45 0.7
CAMERA_POSITION 0 0.5 4
CAMERA_RIGHT 1 0 0
CAMERA_UP 0 1 0
CAMERA_FORWARD 0 0 -1
CAMERA_FOV_X 1.0
AMBIENT_LIGHT 0.08 0.08 0.1

NEW_PRIMITIVE
PLANE 0 1 0
POSITION 0 -1 0
COLOR 0.7 0.7 0.65

NEW_PRIMITIVE
ELLIPSOID 0.9 0.9 0.9
COLOR 0.95 0.95 1.0
DIELECTRIC
IOR 1.5

NEW_PRIMITIVE
BOX 0.4 0.8 0.4
POSITION 1.6 -0.2 -1.5
COLOR 0.2 0.5 0.9

NEW_LIGHT
LIGHT_INTENSITY 0.8 0.8 0.75
LIGHT_DIRECTION -0.4 1 0.6

NEW_LIGHT
LIGHT_INTENSITY 25 22 18
LIGHT_POSITION 0.5 4 2
LIGHT_ATTENUATION 1 0.1 0.25
"""


def test_ray_depth_limits_at_load_and_override(rtc):
    """RAY_DEPTH 62 loads and 63 is refused, in the scene text and through `override` (which then keeps the old value);
    the same for hw2 at 32 and 33."""
    for text, dialect, deepest, message in ((CLOSED_ROOM, 5, 62, "RAY_DEPTH above 62"),
                                            (WHITTED_DEEPEST, 2, 32, "hw2 dialect: RAY_DEPTH above 32")):
        s = rtc.Scene(text=text, device=-1, dialect=dialect)
        assert s.ray_depth == deepest
        with pytest.raises(rtc.RtcError, match=message):
            s.override(ray_depth=deepest + 1)
        assert s.ray_depth == deepest
        s.override(ray_depth=deepest - 1)
        s.override(ray_depth=deepest)
        assert s.ray_depth == deepest
        s.close()
        with pytest.raises(rtc.RtcError, match=message):
            rtc.Scene(text=orclib.with_header(text, ray_depth=deepest + 1), device=-1, dialect=dialect)


def test_whitted_at_the_deepest_ray_depth_in_host_emulation(emu, oracle_lib):
    """hw2 at RAY_DEPTH 32 (course_device.cuh compiled for the host) against the oracle's linear frame."""
    a = orclib.Scene(oracle_lib, text=WHITTED_DEEPEST, dialect=2)
    want, _, rays = a.render_sum(1, 0, 1)
    a.close()
    assert rays > 10 * want.shape[0]   # the glass ball keeps the recursion going
    h = parsed(emu, WHITTED_DEEPEST, dialect=2)
    lin = np.zeros(want.shape, np.float32)
    assert emu.emu_frame_linear(h, lin) == 0
    emu.emu_scene_free(h)
    rel = np.abs(lin - want).max(1) / (np.abs(want).max(1) + 1e-3)
    assert rel.max() <= 1e-5, rel.max()


# ------------------------------------------------------------------------------- CPU: boxes beyond the SAH's infinity
def huge_boxes(half):
    return (HEAD + "NEW_PRIMITIVE\nBOX %g %g %g\nPOSITION 0 0 -5\n\nNEW_PRIMITIVE\nBOX %g %g %g\nPOSITION 10 0 -5\n"
            % ((half,) * 6))


def test_builder_refuses_a_scene_it_cannot_split(rtc):
    """Two boxes of half-size 2e8: every cut, and the leaf too, costs more than the SAH's kInf = 1e18, so the
    reference's builder finds no cut and recurses on the same range for ever.  The library must refuse the scene with
    RTC_ERR_UNSUPPORTED.  A crash would take the test process with it, so the scene is loaded in a child process.
    Half-size 1e8 keeps the leaf cheaper than any cut and loads as one leaf."""
    code = ("import sys\nsys.path.insert(0, %r)\nimport raytracing_course_b200 as rtc\n"
            "try:\n    rtc.Scene(text=sys.stdin.read(), device=-1)\nexcept rtc.RtcError as e:\n    print(e)\n    sys.exit(3)\n"
            % ROOT)
    r = subprocess.run([sys.executable, "-c", code], input=huge_boxes(2e8), capture_output=True, text=True, timeout=300)
    assert r.returncode == 3, (r.returncode, r.stdout[-500:], r.stderr[-500:])
    assert "no cut below 1e18" in r.stdout
    s = rtc.Scene(text=huge_boxes(1e8), device=-1)
    assert s.nnodes == 1
    s.close()


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FALLBACK_SCENES))
def test_fallback_probes_vs_oracle(rtc, oracle_lib, name):
    """RayIntersection (k_traverse) in INDEX mode against REFTREE and the oracle on the rays of the emulation test.  The
    probe shares the render's counters: the fallback ran on the device exactly when the scene has more than 24
    primitives on one ray; at 24 every ray is replayed from its records, 24 at most."""
    from test_gpu_parity import check_hits
    text, nprims = FALLBACK_SCENES[name]
    s = rtc.Scene(text=text, device=0)
    a = orclib.Scene(oracle_lib, text=text)
    o, d = fence_rays(a)
    want = a.intersect(o, d)
    a.close()
    s.reset_counters()
    fast = s.RayIntersection(o, d, rtc.TRAVERSAL_INDEX)
    fallbacks = s.counters()["fallback_rays"]
    slow = s.RayIntersection(o, d, rtc.TRAVERSAL_REFTREE)
    s.close()
    print("%s: %d of %d rays fell back; INDEX != REFTREE on %d, INDEX != oracle on %d, REFTREE != oracle on %d"
          % (name, fallbacks, len(o), (fast[0] != slow[0]).sum(), (fast[0] != want[0]).sum(), (slow[0] != want[0]).sum()))
    assert np.array_equal(fast[0], slow[0])
    check_hits(fast, want, id_agree=1.0)
    check_hits(slow, want, id_agree=1.0)
    if nprims <= K_MAX_RECORDS:
        assert fallbacks == 0
    else:
        assert fallbacks > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fence_25", "triangle_stack_25", "triangle_stack_plane_25"])
def test_fallback_in_render_vs_oracle(rtc, oracle_lib, name):
    """A render in which fallback lanes share warps with replaying lanes over several bounces: sample-exact against
    the oracle (the tolerances of test_render_sample_exact_vs_oracle), with k_traverse as it renders and as it counts
    node visits (set_profiling(count_visits=True) selects the other instantiation)."""
    text, _ = FALLBACK_SCENES[name]
    s = rtc.Scene(text=text, device=0)
    a = orclib.Scene(oracle_lib, text=text)
    want, paths, rays = a.render_sum(9, 2, a.samples)
    a.close()
    for count_visits in (False, True):
        s.set_profiling(count_visits=count_visits)
        s.reset_counters()
        got = s.RenderSum(seed=9, sample_begin=2, sample_count=s.samples).reshape(-1, 3)
        c = s.counters()
        ok = np.isfinite(want).all(1) & np.isfinite(got).all(1)
        rel = np.abs(got - want).max(1) / (np.abs(want).max(1) + 1e-3)
        good = (rel <= 2e-3) & ok
        print("%s count_visits=%d: %d fallback rays of %d, %d node visits, %.5f of the pixels within 2e-3"
              % (name, count_visits, c["fallback_rays"], c["rays"], c["index_node_visits"], good.mean()))
        assert c["paths"] == paths
        assert abs(c["rays"] - rays) <= 1e-3 * rays
        assert c["fallback_rays"] > 0
        assert (c["index_node_visits"] > 0) == count_visits
        assert good.mean() >= 0.99, good.mean()
        squash = lambda x: x / (1.0 + x)
        assert abs(np.median(squash(got[ok])) - np.median(squash(want[ok]))) < 1e-3
    s.close()


@pytest.mark.gpu
def test_hw1_fence_frame_vs_oracle(rtc, oracle_lib):
    """hw1 on the device, 40-box fence: `collect_leaf_hits` gives up on the rays along the axis and the device walks the
    reference tree.  The colours are flat, so the linear frame equals the oracle's exactly.  The 8-bit frame is within 1
    LSB: the device rounds the float product 255 c, the oracle the double one, and for c = 0.7f (the plane's green) the
    two fall on either side of 178.5."""
    text = fence(40)
    s = rtc.Scene(text=text, device=0, dialect=1)
    lin = s.RenderSum(seed=0, sample_count=1).reshape(-1, 3)
    img = s.Render(seed=0)
    s.close()
    a = orclib.Scene(oracle_lib, text=text, dialect=1)
    want_lin = a.render_sum(0, 0, 1)[0]
    want_img = a.frame_u8()
    a.close()
    u8 = np.abs(img.astype(int) - want_img.astype(int)).max(2)
    print("hw1 fence_40: linear frame differs on %d of %d pixels; 8-bit frame off by 1 on %d, by more on %d"
          % ((lin != want_lin).any(1).sum(), len(lin), (u8 == 1).sum(), (u8 > 1).sum()))
    assert same(lin, want_lin)
    assert u8.max() <= 1


@pytest.mark.gpu
def test_leaf_of_64_primitives_probes_vs_oracle(rtc, oracle_lib):
    """The 64-primitive leaf on the device, both traversal modes, against the oracle."""
    from test_gpu_parity import check_hits
    text = ellipsoid_leaf(64)
    s = rtc.Scene(text=text, device=0)
    a = orclib.Scene(oracle_lib, text=text)
    o, d = leaf_rays(a)
    want = a.intersect(o, d)
    a.close()
    fast = s.RayIntersection(o, d, rtc.TRAVERSAL_INDEX)
    slow = s.RayIntersection(o, d, rtc.TRAVERSAL_REFTREE)
    s.close()
    print("leaf_64: INDEX != REFTREE on %d, INDEX != oracle on %d, REFTREE != oracle on %d of %d rays"
          % ((fast[0] != slow[0]).sum(), (fast[0] != want[0]).sum(), (slow[0] != want[0]).sum(), len(o)))
    assert np.array_equal(fast[0], slow[0])
    check_hits(fast, want, id_agree=0.9999)
    check_hits(slow, want, id_agree=0.9999)


@pytest.mark.gpu
def test_paths_reach_the_last_bounce_slot(rtc):
    """RAY_DEPTH 62 in the closed room: the paths really take the 62nd bounce, whose queue slot is the last of 64."""
    s = rtc.Scene(text=CLOSED_ROOM, device=0)
    s.reset_counters()
    s.RenderSum(seed=4, sample_count=s.samples)
    c = s.counters()
    s.close()
    print("closed room: %.3f rays per path" % (c["rays"] / c["paths"]))
    assert c["paths"] == s.width * s.height * s.samples
    assert 61.5 * c["paths"] <= c["rays"] <= 62 * c["paths"]


@pytest.mark.gpu
def test_whitted_at_the_deepest_ray_depth_vs_oracle(rtc, oracle_lib):
    """hw2 at RAY_DEPTH 32 on the device against the oracle's linear frame."""
    s = rtc.Scene(text=WHITTED_DEEPEST, device=0, dialect=2)
    got = s.RenderSum(seed=1, sample_count=1).reshape(-1, 3)
    s.close()
    a = orclib.Scene(oracle_lib, text=WHITTED_DEEPEST, dialect=2)
    want = a.render_sum(1, 0, 1)[0]
    a.close()
    rel = np.abs(got - want).max(1) / (np.abs(want).max(1) + 1e-3)
    print("hw2 depth 32: %d of %d pixels above 1e-4, max %.3g" % ((rel > 1e-4).sum(), len(rel), rel.max()))
    assert (rel <= 1e-4).mean() >= 0.999, (rel > 1e-4).sum()
