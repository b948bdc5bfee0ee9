"""BASELINE.json's full-size configurations on the GPU (streams generated on the device, csrc/gen.cu), ours against what
the reference's own kernels produced through the same C ABI on the same input (tests/golden/reference_parity_b200.npz):
  config 2   36 M-point terrain stream: canonical octree (every node's counters, sorted point / voxel multisets) + Stats
  config 3   350 M-point terrain stream: the deterministic Stats fields, then
  config 5   kernel_render on that octree, 6 cameras x {atomicMin, HQS}: frame digests (tests/reference_golden.py)
  config 4   one GPU's share of the shell stream (250 M points, cube 4096^3): the deterministic Stats fields
"""
import numpy as np
import pytest

import oracle
import reference_golden as golden
from simlod_b200 import SimLOD, camera, data

pytestmark = pytest.mark.gpu
BATCH = 1_000_000


def build(sim, dptr, n, box):
    sim.set_box(*box)
    sim.reset()
    sim.insert_device(dptr, n)
    st = sim.stats()
    assert st.numPointsProcessed == n and st.numPoints == n, (st.numPoints, st.numPointsProcessed, st.dbg)
    return st


def test_config2_36m_stream_canonical_octree_vs_reference_kernels():
    n = 36 * BATCH
    sim = SimLOD(1920, 1080, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=6 << 30, render_blocks_per_sm=3)
    try:
        dptr = sim.device_alloc(n * 16)
        sim.generate(sim.GEN_TERRAIN, dptr, n, 0, n, 7)
        box = ((0.0, 0.0, 0.0), data.TERRAIN_EXTENT)
        st = build(sim, dptr, n, box)
        assert st.dbg == 0
        cn = oracle.canon_from_image(*sim.download_octree())
        ref = golden.octree("config2_36m")
        diffs = oracle.compare_canon(cn, ref, "36M: ours vs reference kernels") + oracle.compare_stats(st, ref.stats)
        assert not diffs, "\n".join(diffs[:10])
    finally:
        sim.close()


def cameras(box_max, w, h):
    cams = [camera.autofocus(box_max, w, h, yaw_offset=k * np.pi / 2) for k in range(4)]
    cams += [camera.orbit_camera(width=w, height=h, **camera.MORRO_BIRD), camera.orbit_camera(width=w, height=h, **camera.MORRO_CLOSE)]
    return cams


def test_config3_350m_stats_and_config5_twelve_frames_vs_reference_kernels():
    n = 350 * BATCH
    # 3 render blocks per SM = the grid the reference's render kernel gets from the occupancy query (EDL tile coverage depends on it)
    sim = SimLOD(1920, 1080, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=24 << 30, render_blocks_per_sm=3)
    try:
        dptr = sim.device_alloc(n * 16)
        sim.generate(sim.GEN_TERRAIN, dptr, n, 0, n, 7)
        box = ((0.0, 0.0, 0.0), data.TERRAIN_EXTENT)
        st = build(sim, dptr, n, box)
        assert st.dbg == 0
        diffs = oracle.compare_stats(st, golden.octree("config3_350m").stats)
        assert not diffs, "\n".join(diffs)
        # config 5: the reference's rasteriser drew the octree our builder made
        for hqs in (0, 1):
            sim.set_settings(useHighQualityShading=hqs, pointSize=1)
            for k, (view, proj) in enumerate(cameras(data.TERRAIN_EXTENT, sim.width, sim.height)):
                sim.set_camera(view, proj)
                sim.render()
                assert sim.stats().numVisibleNodes > 0
                diffs = golden.frame_diffs(golden.frame_digest(sim), "config5/hqs%d/camera%d" % (hqs, k))
                assert not diffs, "\n".join(diffs)
        sim.set_settings(useHighQualityShading=0)
    finally:
        sim.close()


def test_config4_one_gpu_share_of_the_shell_stream_vs_reference_kernels():
    n = 250 * BATCH
    sim = SimLOD(640, 360, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=24 << 30)
    try:
        dptr = sim.device_alloc(n * 16)
        sim.generate(sim.GEN_SHELL, dptr, n, 0, n, 1234)
        box = ((0.0, 0.0, 0.0), (data.SHELL_CUBE,) * 3)
        st = build(sim, dptr, n, box)
        assert st.dbg == 0
        diffs = oracle.compare_stats(st, golden.octree("config4_shell_250m").stats)
        assert not diffs, "\n".join(diffs)
    finally:
        sim.close()
