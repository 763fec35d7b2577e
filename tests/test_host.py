"""CPU: host side of the product (scene parsing, reference-order BVH, C-ABI surface).  No compute
calls: those need a GPU and live in test_gpu_parity.py."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import orclib
from conftest import ROOT, golden, scene_path

SCENES = ["practice5_1", "practice5_2", "lights_mix", "rabbid", "practice5_dragon_10k", "practice5_dragon_100k"]


def test_library_exports_every_declared_symbol(rtc):
    header = open(rtc.HEADER_PATH).read()
    declared = set(re.findall(r"\b(rtc_[a-z0-9_]+)\s*\(", header))
    declared -= {"rtc_status"}
    assert len(declared) >= 30
    lib = ctypes.CDLL(rtc.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), "librtc_b200.so does not export " + name
    assert declared == set(rtc.exported_symbols()), "python binding and header disagree"


def test_no_cpu_fallback(rtc):
    s = rtc.Scene(path=scene_path("practice5_2"), device=-1)
    with pytest.raises(rtc.RtcError, match="no CPU path"):
        s.RayIntersection(np.zeros((1, 3)), np.ones((1, 3)))
    with pytest.raises(rtc.RtcError):
        s.Render()
    with pytest.raises(rtc.RtcError):
        s.mix_distrib.Pdf(np.zeros((1, 3)), np.ones((1, 3)), np.ones((1, 3)))
    s.close()


def test_product_does_not_reference_the_oracle():
    pkg = os.path.join(ROOT, "raytracing-course_b200")
    for dirpath, _, files in os.walk(pkg):
        if os.sep + "build" in dirpath:
            continue
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "rt_oracle" not in text and "liboracle" not in text and "orclib" not in text, f


def test_missing_file_and_bad_device(rtc):
    with pytest.raises(rtc.RtcError, match="cannot open"):
        rtc.Scene(path="/nonexistent/scene.txt", device=-1)
    if rtc.device_count() == 0:
        with pytest.raises(rtc.RtcError, match="not available"):
            rtc.Scene(path=scene_path("practice5_1"), device=0)


@pytest.mark.parametrize("name", SCENES)
def test_host_scene_matches_oracle(rtc, oracle_scenes, name):
    """Primitive order after std::partition + BVH sorts, every primitive field and every
    reference-BVH node (boxes bit-exact, links identical)."""
    s = rtc.Scene(path=scene_path(name), device=-1)
    a = oracle_scenes(name)
    assert [s.width, s.height, s.ray_depth, s.samples, s.nprims, s.nbvh, s.nnodes, s.nlights] == \
           [a.width, a.height, a.ray_depth, a.samples, a.nprims, a.nbvh, a.nnodes, a.nlights]
    assert np.array_equal(s.prim_order(), a.prim_order())
    for x, y in zip(s.prims(), a.prims()):
        assert np.array_equal(x.view(np.uint32) if x.dtype == np.float32 else x, y.view(np.uint32) if y.dtype == np.float32 else y)
    sn, an = s.nodes(), a.nodes()
    assert np.array_equal(sn[0].view(np.uint32), an[0].view(np.uint32))
    assert np.array_equal(sn[1], an[1])
    assert sn[2] == an[2]
    st = s.stats()
    assert st["units"] >= 1 and st["index_nodes"] <= max(st["units"] - 1, 0)
    s.close()


def test_host_scene_matches_reference_golden(rtc):
    g = golden("practice5_dragon_10k_rays")
    s = rtc.Scene(path=scene_path("practice5_dragon_10k"), device=-1)
    tm, data = s.prims()
    assert np.array_equal(tm, g["prim_type_material"])
    assert np.bitwise_xor.reduce(data.view(np.uint32).ravel()) == g["prim_data_crc"][0]
    aabb, links, root = s.nodes()
    crc = np.bitwise_xor.reduce((links.ravel().astype(np.uint64) * np.arange(1, links.size + 1, dtype=np.uint64)) & np.uint64(0xFFFFFFFF))
    assert crc == g["node_links_crc"][0]
    assert np.array_equal(aabb.astype(np.float64).sum(0), g["node_aabb_sum"])
    s.close()


QUIRKY = [
    # attributes before the shape line are reset by it; block ends at blank line
    "DIMENSIONS 8 4\nSAMPLES 2\nRAY_DEPTH 3\nNEW_PRIMITIVE\nCOLOR 1 0 0\nPOSITION 1 2 3\nBOX 1 2 3\nIOR 1.5\n\nNEW_PRIMITIVE\nPLANE 0 1 0\nMETALLIC\n",
    # primitive blocks back to back, without blank lines, and a scene command swallowed after a block
    "DIMENSIONS 4 4\nNEW_PRIMITIVE\nELLIPSOID 1 1 1\nNEW_PRIMITIVE\nTRIANGLE 0 0 0 1 0 0 0 1 0\nEMISSION 1 1 1\nSAMPLES 9\nRAY_DEPTH 4\n",
    # unknown words, stray attribute at scene level, CRLF-free trailing spaces, no trailing newline
    "FOO 1 2\nCOLOR 1 1 1\nDIMENSIONS 3 5  \nBG_COLOR 0.1 0.2 0.3\nCAMERA_FOV_X 1.0\nNEW_PRIMITIVE\nBOX 1 1 1\nROTATION 0 0 0.7071068 0.7071068\nDIELECTRIC",
    # empty scene, planes only
    "",
    "DIMENSIONS 2 2\nNEW_PRIMITIVE\nPLANE 0 0 1\nNEW_PRIMITIVE\nPLANE 1 0 0\nPOSITION 1 0 0\n",
]


@pytest.mark.parametrize("text", QUIRKY)
def test_parser_quirks_match_oracle(rtc, oracle_lib, text):
    s = rtc.Scene(text=text, device=-1)
    raw = text.encode()
    h = oracle_lib.lib.orc_scene_parse(raw, len(raw))
    info = np.zeros(8, np.uint32)
    oracle_lib.lib.orc_scene_info(h, info)
    assert [s.width, s.height, s.ray_depth, s.samples, s.nprims, s.nbvh, s.nnodes, s.nlights] == info.tolist()
    if s.nprims:
        tm = np.zeros((s.nprims, 2), np.int32)
        d = np.zeros((s.nprims, 26), np.float32)
        oracle_lib.lib.orc_scene_prims(h, tm, d)
        stm, sd = s.prims()
        assert np.array_equal(stm, tm)
        assert np.array_equal(sd, d)
    oracle_lib.lib.orc_scene_free(h)
    s.close()


def test_cli_without_gpu_fails_loudly(rtc, tmp_path):
    if rtc.device_count() > 0:
        pytest.skip("GPU present")
    out = str(tmp_path / "should_not_exist.ppm")
    r = subprocess.run([rtc.CLI_PATH, scene_path("practice5_1"), out], capture_output=True, text=True)
    assert r.returncode != 0
    assert "not available" in r.stderr
    assert not os.path.exists(out)
    r = subprocess.run([rtc.CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


def test_host_philox_known_answer(rtc):
    out = rtc.philox4x32_10([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0])
    assert out.tolist() == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_unsupported_scene_is_refused_with_a_message(rtc):
    """More than 64 primitives in one reference BVH leaf (70 coincident ellipsoids) exceeds a documented limit."""
    text = "DIMENSIONS 4 4\nSAMPLES 1\nRAY_DEPTH 1\n" + "NEW_PRIMITIVE\nELLIPSOID 1 1 1\nPOSITION 0 0 0\n\n" * 70
    with pytest.raises(rtc.RtcError, match="more than 64 primitives"):
        rtc.Scene(text=text, device=-1)
    with pytest.raises(rtc.RtcError, match="RAY_DEPTH"):
        rtc.Scene(text="DIMENSIONS 4 4\nRAY_DEPTH 100\nNEW_PRIMITIVE\nBOX 1 1 1\n", device=-1)


# values the reference leaves INDETERMINATE (a missing third argument of POSITION / BOX is never
# written: glm vectors are not zero-initialised); we define them as 0
PARSER_INDETERMINATE = {3: [(0, 8), (1, 16)]}


def test_parser_quirks_match_reference_golden(rtc):
    """The product's scene reader against what the REFERENCE made of the same unusual texts."""
    g = golden("parser_quirks")
    i = 0
    while "text%d" % i in g:
        s = rtc.Scene(text=g["text%d" % i].tobytes(), device=-1)
        assert [s.width, s.height, s.ray_depth, s.samples, s.nprims, s.nbvh, s.nnodes, s.nlights] == g["info%d" % i].tolist(), i
        tm, d = s.prims()
        assert np.array_equal(tm, g["tm%d" % i]), i
        want = g["data%d" % i].copy()
        for r, c in PARSER_INDETERMINATE.get(i, []):
            want[r, c] = d[r, c]
        assert np.array_equal(d, want), (i, np.argwhere(d != want).tolist())
        s.close()
        i += 1
    assert i == 4


def test_parser_number_formats_match_reference_golden(rtc):
    """Number formats at the edge of the reader's fast path (plain decimals via std::from_chars, everything else via
    operator>>): signs, bare dots, exponents, hex, inf / nan, trailing garbage, commas, over- and underflow, CRLF --
    against what the REFERENCE made of the same texts (tools/make_golden.py parser_numbers)."""
    g = golden("parser_numbers")
    i = 0
    while "text%d" % i in g:
        s = rtc.Scene(text=g["text%d" % i].tobytes(), device=-1)
        assert [s.width, s.height, s.ray_depth, s.samples, s.nprims, s.nbvh, s.nnodes, s.nlights] == g["info%d" % i].tolist(), i
        tm, d = s.prims()
        assert np.array_equal(tm, g["tm%d" % i]), i
        assert np.array_equal(d, g["data%d" % i]), (i, np.argwhere(d != g["data%d" % i]).tolist())
        s.close()
        i += 1
    assert i == 2


def test_bench_configs_and_reference_arm(tmp_path):
    """bench.py: every BASELINE.json configuration resolves to its scene / size, and the reference arm prints the
    contract's JSON line (a tiny sample here: 8x8 pixels, 1 spp of the 10k dragon through the compiled reference, or
    through the oracle's port of it where oracle/_ref has not been built)."""
    import json
    import subprocess
    import sys
    sys.path.insert(0, ROOT)
    import bench
    import orclib

    class A:
        scene = ""; width = -1; height = -1; spp = -1
    want = {1: "practice5_1", 2: "practice5_dragon_10k", 3: "practice5_dragon_100k", 4: "practice5_dragon_100k_glass",
            5: "practice5_dragon_100k_metal"}
    for c, name in want.items():
        a = A(); a.config = c
        cfg = bench.resolve_config(a)
        assert cfg["scene"] == name
    a = A(); a.config = 5
    assert (bench.resolve_config(a)["width"], bench.resolve_config(a)["height"], bench.resolve_config(a)["spp"]) == (3840, 2160, 1024)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "2", "--steps", "1",
                        "--warmup", "0", "--ref-width", "8", "--ref-height", "8", "--ref-spp", "1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "Mpaths/s" and line["value"] > 0
    kind = "reference" if orclib.have_ref() else "port"
    assert line["config"]["workload"] == "practice5_dragon_10k" and line["cpu_baseline"]["kind"] == kind
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True
