"""CPU-only: ABI layouts, the C-ABI library loads and exports every declared symbol, host logic
fails loudly without a device. No compute is executed here."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import HAVE_GPU, ROOT
from simlod_b200 import api, camera, data


def test_abi_header_compiles_as_c_and_cpp(tmp_path):
    src = tmp_path / "abi.c"
    src.write_text('#include "simlod_abi.h"\n#include "simlod_b200.h"\nint main(void){return 0;}\n')
    for cc in (["gcc", "-x", "c"], ["g++", "-x", "c++"]):
        subprocess.check_call(cc + ["-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])


def test_ctypes_mirrors_match_reference_layout():
    # sizes/offsets of SURVEY.md §7.1 (probed from the reference headers)
    assert C.sizeof(api.Uniforms) == 480
    assert api.Uniforms.transform.offset == 208
    assert api.Uniforms.transform_updateBound.offset == 272
    assert api.Uniforms.persistentBufferCapacity.offset == 400
    assert api.Uniforms.boxMin.offset == 424 and api.Uniforms.boxMax.offset == 436
    assert api.Uniforms.useHighQualityShading.offset == 460
    assert api.Uniforms.minNodeSize.offset == 464 and api.Uniforms.pointSize.offset == 468
    assert C.sizeof(api.Stats) == 112
    assert api.Stats.numNodes.offset == 4 and api.Stats.batchletIndex.offset == 76
    assert api.Stats.numPointsProcessed.offset == 80 and api.Stats.numAllocatedChunks.offset == 88
    assert api.Stats.chunkPoolSize.offset == 96 and api.Stats.memCapacityReached.offset == 108
    assert api.POINT_DTYPE.itemsize == 16


def test_library_exports_every_declared_symbol():
    lib = api.load_library()
    header = open(os.path.join(ROOT, "include", "simlod_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(simlod_[a-z0-9_]+)\s*\(", header)))
    assert declared == sorted(api.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    nm = subprocess.check_output(["nm", "-D", "--defined-only", api.LIB_PATH], text=True)
    exported = set(re.findall(r" T (simlod_[a-z0-9_]+)", nm))
    assert set(declared) <= exported


def test_cubins_are_sm100a_and_export_reference_kernel_names():
    for prog, kernel in (("construct", "kernel_construct"), ("render", "kernel_render"), ("reset", "kernel")):
        path = os.path.join(ROOT, "simlod_b200", "cubin", "simlod_%s.cubin" % prog)
        out = subprocess.check_output(["cuobjdump", "-elf", path], text=True, stderr=subprocess.STDOUT)
        assert "sm_100a" in out or "SM100a" in out or "EF_CUDA_SM100" in out, out[:400]
        syms = subprocess.check_output(["cuobjdump", "-symbols", path], text=True, stderr=subprocess.STDOUT)
        assert re.search(r"STT_FUNC\s+STB_GLOBAL\s+\S+\s+%s\b" % kernel, syms) or (" %s" % kernel) in syms


@pytest.mark.skipif(HAVE_GPU, reason="only meaningful without a device")
def test_product_fails_loudly_without_a_device():
    with pytest.raises(api.SimlodError) as e:
        api.SimLOD(64, 64)
    assert "no CPU path" in str(e.value) or "CUDA" in str(e.value)


def test_camera_matches_glm_conventions():
    p = camera.perspective(np.pi / 3, 16 / 9, 0.1, 2e6)
    assert p[3, 2] == -1.0 and p[3, 3] == 0.0
    assert np.isclose(p[1, 1], 1.0 / np.tan(np.pi / 6))
    assert np.isclose(p[0, 0], p[1, 1] / (16 / 9))
    w = camera.orbit_world(0.0, 0.0, 10.0, (1.0, 2.0, 3.0))
    # yaw = pitch = 0: camera sits `radius` along -y of the target (flip maps +z_cam to -y), looking along +y
    assert np.allclose(w @ np.array([0, 0, 0, 1.0]), [1.0, -8.0, 3.0, 1.0])
    view, proj = camera.autofocus((1024, 1024, 1024), 1920, 1080)
    assert np.allclose(view @ np.linalg.inv(view), np.eye(4))


def test_generators_are_counter_based():
    a, mn, mx = data.uniform_cube(5000)
    b, _, _ = data.uniform_cube(1000, first=4000)
    assert (a[4000:] == b).all()
    assert a["x"].max() < 1024 and a["x"].min() >= 0
    t, _, ext = data.terrain(200_000)
    t2, _, _ = data.terrain(200_000, first=150_000, count=1000)
    assert (t[150_000:151_000] == t2).all()
    for ax, e in zip("xyz", ext):
        assert t[ax].min() >= 0 and t[ax].max() < e
    s, _, cube = data.shell(100_000)
    r = np.sqrt(((np.stack([s["x"], s["y"], s["z"]], 1).astype(np.float64) - cube[0] / 2) ** 2).sum(1))
    assert abs(r - 1800).max() < 0.3


def test_abi_matches_the_reference_headers_field_by_field(tmp_path):
    """tests/native/abi_layout.cu prints size and offset of every field of include/simlod_abi.h's records and the
    constants; built against the reference's OWN HostDeviceInterface.h / structures.cuh it printed
    tests/golden/reference_abi_layout.txt. Both must agree line by line."""
    import reference_golden as golden
    exe = str(tmp_path / "abi_layout")
    subprocess.check_call(["g++", "-std=c++17", "-x", "c++", "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "native", "abi_layout.cu")])
    ours = subprocess.check_output([exe], text=True).splitlines()
    ref = open(golden.ABI_LAYOUT).read().splitlines()
    assert len(ours) == len(ref) == 90
    diffs = [(a, b) for a, b in zip(ours, ref) if a != b]
    assert not diffs, diffs
