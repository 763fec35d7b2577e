"""CPU: the per-pixel candidate lists camera rays are resolved from (rt_device.cuh pixel_beam / pixel_candidates), compiled
for the host by tests/host_emul/beam_emul.cpp.  For random pixels and jitters, including u = 0 and u = 1 - 2^-24 (the
extremes of u01) and hw3's half-pixel offset: every leaf the ray's own index traversal reaches is in its pixel's list
(or the pixel is marked for the index traversal), and the list gives the id the index traversal gives."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, scene_path
from test_limits import fence, triangle_stack

EMU_DIR = os.path.join(ROOT, "tests", "host_emul")
CSRC = os.path.join(ROOT, "raytracing-course_b200", "csrc")
TRAVERSE = 0xFFFFFFFF
U_MAX = np.float32(0xFFFFFF / 16777216.0)   # the largest jitter u01 makes


@pytest.fixture(scope="module")
def beam():
    objs = [os.path.join(CSRC, "build", "scene_load.o"), os.path.join(CSRC, "build", "bvh_build.o")]
    if not all(os.path.exists(o) for o in objs):
        pytest.skip("product objects not built")
    cuda_inc = "/usr/local/cuda/include"
    if not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("CUDA headers not found")
    so = os.path.join(EMU_DIR, "libbeam_emul.so")
    srcs = [os.path.join(EMU_DIR, "beam_emul.cpp"), os.path.join(EMU_DIR, "emul.cpp"), os.path.join(CSRC, "rt_device.cuh"),
            os.path.join(CSRC, "device_scene.h")]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(p) for p in srcs + objs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off",
                               "-I" + cuda_inc, "-I" + CSRC, "-I" + os.path.join(ROOT, "include"), srcs[0]] + objs + ["-o", so])
    L = C.CDLL(so)
    L.emu_scene_load.restype = C.c_void_p
    L.emu_scene_load.argtypes = [C.c_char_p]
    L.emu_scene_parse_dialect.restype = C.c_void_p
    L.emu_scene_parse_dialect.argtypes = [C.c_char_p, C.c_long, C.c_int]
    L.emu_scene_free.argtypes = [C.c_void_p]
    u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
    L.emu_camera_lists.argtypes = [C.c_void_p, C.c_long, u32p, np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS"),
                                   np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")]
    L.emu_camera_list_lengths.argtypes = [C.c_void_p, u32p]
    return L


def scene_text(name):
    """(text, dialect): the fallback scenes of test_limits, hw3 fixtures (half-pixel offset), scenes under scenes/"""
    if name == "fence_25":
        return fence(25), 5
    if name == "triangle_stack_25":
        return triangle_stack(25), 5
    if name.startswith("hw3_"):
        g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        return bytes(g["text"]).decode(), int(g["dialect"])
    return open(scene_path(name)).read(), 5


def load(L, name):
    text, dialect = scene_text(name)
    b = text.encode()
    h = L.emu_scene_parse_dialect(b, len(b), dialect)
    assert h
    return h


def dims(text):
    for line in text.splitlines():
        if line.startswith("DIMENSIONS"):
            return int(line.split()[1]), int(line.split()[2])
    raise AssertionError("no DIMENSIONS")


SCENES = ["practice5_dragon_10k", "practice5_dragon_100k", "lights_mix", "rabbid", "fence_25", "triangle_stack_25",
          "hw3_course_sample3", "hw3_course_sample6"]


@pytest.mark.parametrize("name", SCENES)
def test_lists_hold_every_reached_leaf_and_give_the_same_id(beam, name):
    h = load(beam, name)
    try:
        w, hh = dims(scene_text(name)[0])
        npix = w * hh
        lengths = np.zeros(npix, np.uint32)
        beam.emu_camera_list_lengths(h, lengths)
        rng = np.random.default_rng(7)
        # random pixels plus the pixels with the longest lists; every pixel once at each corner of its jitter square
        pix = np.concatenate([rng.integers(0, npix, 3000), np.argsort(np.where(lengths == TRAVERSE, 0, lengths))[-200:]])
        pix = pix.astype(np.uint32)
        corners = np.array([[0, 0], [U_MAX, 0], [0, U_MAX], [U_MAX, U_MAX]], np.float32)
        u = np.concatenate([rng.random((pix.size, 2), dtype=np.float32).clip(0, U_MAX)] + [np.tile(c, (pix.size, 1)) for c in corners])
        pix = np.tile(pix, 5)
        out = np.zeros((pix.size, 4), np.int32)
        beam.emu_camera_lists(h, pix.size, pix, np.ascontiguousarray(u), out)
        listed = out[:, 0].view(np.uint32) != TRAVERSE
        assert (out[listed, 1] == 0).all(), "a leaf the ray's traversal reaches is missing from its pixel's list"
        assert np.array_equal(out[listed, 2], out[listed, 3])
        assert (out[:, 0].view(np.uint32)[listed] <= 24).all()
        if name in ("fence_25", "triangle_stack_25"):
            # more than kMaxRecords leaves along the rays: those pixels keep the index traversal and its fallback
            assert (lengths == TRAVERSE).any()
        elif not name.startswith("hw3_"):   # (a scene with a handful of primitives may have no index tree)
            assert listed.mean() > 0.9
    finally:
        beam.emu_scene_free(h)
