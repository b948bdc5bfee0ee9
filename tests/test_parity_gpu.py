"""GPU parity tests (run on the B200 box with -m gpu). Everything goes through the C ABI.

Three-way comparison on the same inputs:
  ours (built-in sm_100a cubins)  vs  CPU oracle (oracle/oracle.cpp)  vs  what the reference's own
  kernels produced on a B200 (tests/golden/reference_parity_b200.npz, see tests/reference_golden.py).
Integer/byte results are compared bit-exactly on the canonical form (DESIGN.md §3); a frame is compared
through its digest (visibility counters and flags, depth words, whole framebuffer and surface), recorded
with the reference's rasteriser drawing the octree our builder made.
"""
import numpy as np
import pytest

import oracle
import reference_golden as golden
from simlod_b200 import SimLOD, camera, data

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sim():
    # 3 render blocks per SM = the grid the reference's own kernel gets from the occupancy query on
    # sm_100 (72 registers); EDL tile coverage depends on the grid size (render.cu:1273)
    s = SimLOD(1920, 1080, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=12 << 30, render_blocks_per_sm=3)
    yield s
    s.close()


def build_gpu(sim, batches, box):
    sim.set_box(*box)
    sim.reset()
    sim.insert_batches(batches)
    stats = sim.stats()
    canon = oracle.canon_from_image(*sim.download_octree())
    return stats, canon


def build_oracle(batches, box, rcp=0.0):
    o = oracle.Oracle(box[0], box[1], rcp)
    for b in batches:
        o.add_batch(b)
    return o


def assert_same_octree(stats_a, canon_a, stats_b, canon_b, label):
    diffs = oracle.compare_canon(canon_a, canon_b, label) + oracle.compare_stats(stats_a, stats_b)
    assert not diffs, "\n".join(diffs)


def assert_reference_octree(stats, canon, key, label="ours vs reference kernels"):
    ref = golden.octree(key)
    assert_same_octree(stats, canon, ref.stats, ref, label)
    return ref


def assert_reference_frame(sim, key, canon=None):
    diffs = golden.frame_diffs(golden.frame_digest(sim, canon), key)
    assert not diffs, "\n".join(diffs)


def split(points, sizes):
    out, s = [], 0
    for n in sizes:
        out.append(points[s:s + n])
        s += n
    assert s == len(points)
    return out


# ---- builder --------------------------------------------------------------------------------------

def test_config1_uniform_1m_single_batch_vs_oracle(sim):
    pts, mn, mx = data.uniform_cube(1_000_000)
    st, cn = build_gpu(sim, [pts], (mn, mx))
    o = build_oracle([pts], (mn, mx))
    assert st.numNodes == 73 and st.numInner == 9 and st.numLeaves == 64 and st.dbg == 0
    assert_same_octree(st, cn, o.stats(), o.canon(), "ours vs oracle")
    assert o.check_voxel_colors(cn) == 0


def test_config1_uniform_1m_single_batch_vs_reference_kernels(sim):
    # (that the reference's voxel colours pass oracle.check_voxel_colors was checked when the golden data was recorded)
    pts, mn, mx = data.uniform_cube(1_000_000)
    st, cn = build_gpu(sim, [pts], (mn, mx))
    ref = assert_reference_octree(st, cn, "config1_uniform_1m")
    o = build_oracle([pts], (mn, mx))
    assert_same_octree(ref.stats, ref, o.stats(), o.canon(), "reference kernels vs oracle")


TERRAIN_N = 3_300_000


def terrain_batches():
    pts, mn, mx = data.terrain(TERRAIN_N)
    # ragged stream: full batches, a tiny one, an empty one, a final partial one
    sizes = [1_000_000, 1_000_000, 7, 0, 900_000, TERRAIN_N - 2_900_007]
    return split(pts, sizes), (mn, mx)


def test_streamed_ragged_batches_vs_oracle(sim):
    batches, box = terrain_batches()
    st, cn = build_gpu(sim, batches, box)
    rcp = float(sim.device_rcp(4800.0))        # cube size 4800 is not a power of two: MUFU.RCP comes from the device
    o = build_oracle(batches, box, rcp)
    assert st.dbg == 0 and st.numPointsProcessed == TERRAIN_N and st.numPoints == TERRAIN_N
    assert_same_octree(st, cn, o.stats(), o.canon(), "ours vs oracle")
    assert o.check_voxel_colors(cn) == 0


def test_streamed_ragged_batches_vs_reference_kernels(sim):
    batches, box = terrain_batches()
    st, cn = build_gpu(sim, batches, box)
    assert_reference_octree(st, cn, "streamed_ragged_terrain")


def test_small_batches_grow_a_leaf_root_then_split(sim):
    # the root is a leaf that owns an occupancy grid (reset.cu:69); its grid is wiped when it splits
    pts, mn, mx = data.uniform_cube(120_000, size=64.0, seed=5)
    batches = split(pts, [20_000, 20_000, 10_000, 1, 30_000, 39_999])
    st, cn = build_gpu(sim, batches, (mn, mx))
    o = build_oracle(batches, (mn, mx))
    assert_same_octree(st, cn, o.stats(), o.canon(), "ours vs oracle")
    assert o.check_voxel_colors(cn) == 0


def test_small_batches_vs_reference_kernels(sim):
    pts, mn, mx = data.uniform_cube(120_000, size=64.0, seed=5)
    batches = split(pts, [20_000, 20_000, 10_000, 1, 30_000, 39_999])
    st, cn = build_gpu(sim, batches, (mn, mx))
    assert_reference_octree(st, cn, "small_batches")


def test_leaf_capacity_is_inclusive_and_out_of_box_points_are_mirrored(sim):
    # 50 000 points in one octant leaf do not split it; the 50 001st does (voxels.cu:211-217).
    rng = np.random.default_rng(3)
    n = 200_000
    xyz = rng.random((n, 3), dtype=np.float32) * np.float32(32.0)
    from simlod_b200 import make_points
    pts = make_points(xyz, np.arange(n, dtype=np.uint32) | np.uint32(0xFF000000))
    # outliers: on the max face (X = 2^20 wraps to child bit 0), beyond it, negative (saturates to 0)
    pts["x"][:4] = [32.0, 40.0, -5.0, 31.999998]
    pts["y"][4:6] = [32.0, -0.0]
    batches = split(pts, [50_000, 1, 49_999, 100_000])
    box = ((0.0, 0.0, 0.0), (32.0, 32.0, 32.0))
    st, cn = build_gpu(sim, batches, box)
    o = build_oracle(batches, box)
    assert_same_octree(st, cn, o.stats(), o.canon(), "ours vs oracle")


def test_nonzero_box_min_and_anisotropic_box(sim):
    pts, _, _ = data.uniform_cube(300_000, size=256.0, seed=11)
    pts["x"] += np.float32(100.0)
    pts["y"] = pts["y"] * np.float32(0.5) + np.float32(-20.0)
    box = ((100.0, -20.0, 0.0), (356.0, 108.0, 256.0))     # cube edge = max extent = 256
    st, cn = build_gpu(sim, [pts], box)
    o = build_oracle([pts], box)
    assert_same_octree(st, cn, o.stats(), o.canon(), "ours vs oracle")


# ---- rasteriser -------------------------------------------------------------------------------------

def cameras(box_size, w, h):
    yield "autofocus", camera.autofocus(box_size, w, h)
    yield "autofocus+pi/2", camera.autofocus(box_size, w, h, yaw_offset=np.pi / 2)
    r = float(np.linalg.norm(box_size))
    yield "close", camera.orbit_camera(0.4, -0.3, r * 0.08, (box_size[0] * 0.55, box_size[1] * 0.45, box_size[2] * 0.3), w, h)
    yield "far", camera.orbit_camera(-2.0, -0.9, r * 6.0, (box_size[0] * 0.5, box_size[1] * 0.5, 0.0), w, h)
    yield "inside", camera.orbit_camera(2.2, 0.1, r * 0.01, (box_size[0] * 0.5, box_size[1] * 0.5, box_size[2] * 0.5), w, h)


def scribble_like_another_renderer(sim):
    """Overwrite the head of the render buffer the way the reference's kernel_render uses it between our frames: as
    scratch for copies of the octree's Node records (render.cu:1108-1123 keeps up to 100 000 of them there)."""
    st = sim.stats()
    nodes = sim.memcpy_dtoh(sim.buffers().nodes, st.numNodes * 152)
    reps = -(-31_200_144 // nodes.nbytes)
    sim.memcpy_htod(sim.buffers().renderbuffer, np.tile(nodes, reps)[:31_200_144])


@pytest.mark.parametrize("hqs", [0, 1])
@pytest.mark.parametrize("dataset", ["uniform", "terrain"])
def test_framebuffer_bit_exact_vs_reference_kernel(sim, dataset, hqs):
    if dataset == "uniform":
        pts, mn, mx = data.uniform_cube(1_000_000)
        batches = [pts]
    else:
        pts, mn, mx = data.terrain(4_000_000)
        batches = list(data.batches(pts))
    _, cn = build_gpu(sim, batches, (mn, mx))
    sim.set_settings(useHighQualityShading=hqs, pointSize=1)
    for name, (view, proj) in cameras(mx, sim.width, sim.height):
        sim.set_camera(view, proj)
        sim.render()
        assert_reference_frame(sim, "framebuffer/%s/hqs%d/%s" % (dataset, hqs, name), cn)
    sim.set_settings(useHighQualityShading=0)


LOD_COLOUR_SETTINGS = (dict(pointSize=2), dict(pointSize=1, colorByLOD=1), dict(pointSize=3, useHighQualityShading=1),
                       dict(colorByNode=1), dict(colorByNode=1, colorByLOD=1), dict(colorByNode=1, useHighQualityShading=1))   # render.cu:73-78


def test_framebuffer_point_size_2_and_lod_colours(sim):
    pts, mn, mx = data.terrain(2_000_000)
    _, cn = build_gpu(sim, list(data.batches(pts)), (mn, mx))
    view, proj = camera.autofocus(mx, sim.width, sim.height)
    sim.set_camera(view, proj)
    for k, settings in enumerate(LOD_COLOUR_SETTINGS):
        sim.set_settings(pointSize=1, colorByLOD=0, colorByNode=0, useHighQualityShading=0)
        sim.set_settings(**settings)
        sim.render()
        assert_reference_frame(sim, "lod_colours/%d" % k, cn)
    sim.set_settings(pointSize=1, colorByLOD=0, colorByNode=0, useHighQualityShading=0)


def test_framebuffer_with_frozen_visibility_transform(sim):
    # settings.doUpdateVisibility off (main.cpp:300-306): the LOD cut keeps the bound transform of the previous view
    # (transform_updateBound, render.cu:792-852) while the samples are splatted with the new one (transform, render.cu:62)
    pts, mn, mx = data.terrain(2_000_000)
    _, cn = build_gpu(sim, list(data.batches(pts)), (mn, mx))
    sim.set_settings(pointSize=1, colorByLOD=0, useHighQualityShading=0)
    r = float(np.linalg.norm(mx))
    far = camera.orbit_camera(-2.0, -0.9, r * 6.0, (mx[0] * 0.5, mx[1] * 0.5, 0.0), sim.width, sim.height)
    close = camera.orbit_camera(0.4, -0.3, r * 0.08, (mx[0] * 0.55, mx[1] * 0.45, mx[2] * 0.3), sim.width, sim.height)
    for hqs in (0, 1):
        sim.set_settings(useHighQualityShading=hqs)
        sim.set_camera(*far)
        sim.set_camera(*close, update_visibility=False)
        sim.render()
        frozen_stats, frozen_fb = sim.stats(), sim.framebuffer()
        assert_reference_frame(sim, "frozen/hqs%d/frozen" % hqs, cn)
        assert frozen_stats.numVisibleVoxels > 0 and frozen_stats.numVisiblePoints == 0      # the far cut, seen from close
        sim.set_camera(*close)
        sim.render()
        moved_fb = sim.framebuffer()
        assert_reference_frame(sim, "frozen/hqs%d/moved" % hqs, cn)
        assert (frozen_fb != moved_fb).any()
    sim.set_settings(useHighQualityShading=0)


def cache_counters(sim):
    """RCtl::cacheHits / cacheWalks of the last frame (render.cu: lists served from the chunk-list cache / walked)."""
    c = sim.memcpy_dtoh(sim.buffers().renderbuffer + 40, 8).view(np.uint32)
    return int(c[0]), int(c[1])


def test_chunk_list_cache_is_only_a_hint(sim):
    """The rasteriser keeps the chunk pointers of drawn nodes across frames and verifies them against the octree before
    use. Frames must equal the reference kernel's whatever happens between them: growth of the lists, a reset followed by
    a different octree at the same addresses, and another render kernel using the buffer as scratch."""
    pts, mn, mx = data.terrain(5_000_000)
    batches = list(data.batches(pts))
    sim.set_settings(pointSize=1, colorByLOD=0, colorByNode=0, useHighQualityShading=0)
    view, proj = camera.autofocus(mx, sim.width, sim.height)
    sim.set_camera(view, proj)

    def same_as_reference(label):
        sim.render()
        fb = sim.framebuffer()
        assert_reference_frame(sim, "chunk_cache/" + label)
        scribble_like_another_renderer(sim)
        return fb

    build_gpu(sim, batches[:3], (mn, mx))
    a = same_as_reference("first frame")
    sim.render(); sim.render()
    hits, walks = cache_counters(sim)
    assert hits > 0 and walks == 0, (hits, walks)                        # second frame in a row: every list comes from the cache
    assert (sim.framebuffer() == a).all()
    same_as_reference("after another kernel used the buffer")           # its scratch overwrote ours: verified, rebuilt
    # the lists grow: two more batches into the same octree
    for b in batches[3:]:
        sim.upload_batch(b)
    while sim.stats().batchletIndex < len(batches):
        sim.update_octree()
    sim.render(); sim.render()
    same_as_reference("after growth")
    # a reset and a different octree (other points, same heap addresses)
    other, _, _ = data.terrain(3_000_000, seed=11)
    sim.render()
    build_gpu(sim, list(data.batches(other)), (mn, mx))
    b_ = same_as_reference("after a reset")
    assert (a != b_).any()
    # HQS reads the same items
    sim.set_settings(useHighQualityShading=1)
    sim.render()
    same_as_reference("hqs")
    sim.set_settings(useHighQualityShading=0)


def test_framebuffer_vs_cpu_oracle_rasteriser():
    # 320x176: fewer 16x16 tiles than blocks, so the EDL pass covers no tile and the framebuffer is the raw splat
    s = SimLOD(320, 176, persistent_bytes=2 << 30)
    try:
        pts, mn, mx = data.uniform_cube(400_000, size=512.0, seed=9)
        s.set_box(mn, mx)
        s.reset()
        s.insert_batches([pts])
        canon = oracle.canon_from_image(*s.download_octree())
        view, proj = camera.autofocus(mx, 320, 176)
        s.set_camera(view, proj)
        s.render()
        fb = s.framebuffer()
        st = s.stats()
        fb_cpu, rs, _ = canon.render(s.uniforms_bytes(), 320, 176)
        assert rs.numVisibleNodes == st.numVisibleNodes and rs.numVisiblePoints == st.numVisiblePoints
        # 1/w is MUFU.RCP on the device and a correctly rounded reciprocal on the CPU: a sample can land in the
        # neighbouring pixel when its coordinate sits within 1 ulp of a pixel boundary
        mismatch = (fb != fb_cpu).mean()
        assert mismatch < 2e-3, mismatch
    finally:
        s.close()


def test_render_is_idempotent_and_does_not_modify_the_octree(sim):
    pts, mn, mx = data.uniform_cube(500_000, size=128.0, seed=2)
    st, cn = build_gpu(sim, [pts], (mn, mx))
    view, proj = camera.autofocus(mx, sim.width, sim.height)
    sim.set_camera(view, proj)
    sim.render(); a = sim.framebuffer()
    sim.render(); b = sim.framebuffer()
    assert (a == b).all()
    cn2 = oracle.canon_from_image(*sim.download_octree())
    assert not oracle.compare_canon(cn, cn2)


# ---- BASELINE.json full size (configs[1]: 36 M points streamed in 1 M-point batches): size-independent properties ----

def test_full_size_36m_stream_invariants(sim):
    K = 36
    batches, mn, mx = data.terrain_batches(K, list(range(K)))
    sim.set_box(mn, mx)
    sim.reset()
    # two ragged batches in the middle of the stream, the rest full
    stream = batches[:10] + [batches[10][:123_457], batches[10][123_457:]] + batches[11:]
    n = sum(len(b) for b in stream)
    for b in stream:
        sim.upload_batch(b)
    while sim.stats().batchletIndex < len(stream):
        sim.update_octree()
    st = sim.stats()
    assert st.dbg == 0 and st.memCapacityReached == 0
    assert st.numPointsProcessed == n == K * 1_000_000 and st.numPoints == n and st.batchletIndex == len(stream)
    nodes = sim.memcpy_dtoh(sim.buffers().nodes, st.numNodes * 152)
    rec = np.frombuffer(nodes.tobytes(), dtype=np.dtype({
        "names": ["child0", "counter", "numPoints", "level", "X", "Y", "Z", "grid", "points", "voxelChunks", "numVoxels", "numVoxelsStored"],
        "formats": ["<u8", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u8", "<u8", "<u8", "<u4", "<u4"],
        "offsets": [0, 64, 68, 72, 76, 80, 84, 120, 128, 136, 144, 148], "itemsize": 152}))
    leaf = rec["child0"] == 0
    inner = ~leaf
    assert st.numNodes == len(rec) == 1 + 8 * int(inner.sum()) and st.numInner == int(inner.sum()) and st.numLeaves == int(leaf.sum())
    assert int(rec["numPoints"][leaf].sum()) == n and (rec["numPoints"][inner] == 0).all() and (rec["points"][inner] == 0).all()
    assert (rec["numPoints"][leaf] <= 50_000).all() and (rec["counter"][leaf] == rec["numPoints"][leaf]).all()
    assert (rec["counter"][inner] > 50_000).all()                      # an inner node is a leaf that crossed the capacity once
    assert (rec["grid"][inner] != 0).all() and (rec["grid"][leaf & (rec["level"] > 0)] == 0).all()
    assert (rec["numVoxels"] == rec["numVoxelsStored"]).all() and (rec["numVoxels"][leaf & (rec["level"] > 0)] == 0).all()
    assert (rec["numVoxels"][inner & (rec["level"] > 0)] <= 128 ** 3).all()
    # keys are unique and every non-root node's parent exists and is inner
    keys = (rec["level"].astype(np.uint64) << np.uint64(60)) | (rec["X"].astype(np.uint64) << np.uint64(40)) | (rec["Y"].astype(np.uint64) << np.uint64(20)) | rec["Z"].astype(np.uint64)
    assert len(np.unique(keys)) == len(keys)
    nz = rec["level"] > 0
    pkeys = ((rec["level"][nz] - 1).astype(np.uint64) << np.uint64(60)) | ((rec["X"][nz] >> 1).astype(np.uint64) << np.uint64(40)) | ((rec["Y"][nz] >> 1).astype(np.uint64) << np.uint64(20)) | (rec["Z"][nz] >> 1).astype(np.uint64)
    assert np.isin(pkeys, keys[inner]).all()
    # chunk / heap accounting identities (DESIGN.md §3)
    chunks_points = int(((rec["numPoints"][leaf] + 999) // 1000).sum())
    chunks_voxels = int(((rec["numVoxels"] + 999) // 1000).sum())
    assert st.numAllocatedChunks == chunks_points == st.numChunksPoints and st.chunkPoolSize >= st.numAllocatedChunks
    assert st.allocatedBytes_persistent == 16 + 262160 * int(inner.sum()) + 16032 * (st.chunkPoolSize + chunks_voxels)
    assert st.numVoxels == int(rec["numVoxels"][inner].sum())
    # rendering the full-size octree twice gives the same framebuffer, and a sane one
    view, proj = camera.orbit_camera(width=sim.width, height=sim.height, **camera.MORRO_BIRD)
    sim.set_camera(view, proj)
    sim.render(); a = sim.framebuffer(); s1 = sim.stats()
    sim.render(); b = sim.framebuffer()
    assert (a == b).all() and s1.numVisibleNodes > 0
    drawn = (a >> np.uint64(32)) != np.uint64(0x7f800000)
    assert 0.05 < drawn.mean() <= 1.0


def test_reference_launch_shape_one_block_per_sm():
    """The unmodified reference host launches kernel_construct with numSMs blocks (main.cpp:370-371): the drop-in
    must produce the same octree at that shape (and at any other cooperative grid)."""
    pts, mn, mx = data.terrain(2_200_000)
    batches = split(pts, [1_000_000, 999, 1_000_000, 199_001])
    o = build_oracle(batches, (mn, mx), 0.0)   # rcp filled below
    for per_sm in (1, 2):
        s = SimLOD(640, 360, persistent_bytes=4 << 30, construct_blocks_per_sm=per_sm, render_blocks_per_sm=per_sm)
        try:
            assert s.launch_info()["construct_blocks"] == per_sm * s.launch_info()["num_sms"]
            rcp = float(s.device_rcp(4800.0))
            o = build_oracle(batches, (mn, mx), rcp)
            s.set_box(mn, mx)
            s.reset()
            s.insert_batches(batches)
            st = s.stats()
            cn = oracle.canon_from_image(*s.download_octree())
            assert st.dbg == 0
            assert_same_octree(st, cn, o.stats(), o.canon(), "ours at %d block(s)/SM vs oracle" % per_sm)
            assert o.check_voxel_colors(cn) == 0
            view, proj = camera.autofocus(mx, 640, 360)
            s.set_camera(view, proj)
            s.render()
            assert s.stats().numVisibleNodes > 0
        finally:
            s.close()


def test_shell_and_incoherent_streams_vs_oracle(sim):
    # config-4 geometry (sphere shell in latitude/longitude tile order) and a spatially incoherent stream
    # (uniform random: many leaves fill at the same rate and split in the same batch)
    pts, mn, mx = data.shell(2_400_000)
    batches = list(data.batches(pts))
    st, cn = build_gpu(sim, batches, (mn, mx))
    o = build_oracle(batches, (mn, mx))
    assert st.dbg == 0
    assert_same_octree(st, cn, o.stats(), o.canon(), "shell: ours vs oracle")
    assert o.check_voxel_colors(cn) == 0

    pts, mn, mx = data.uniform_cube(3_000_000, size=2048.0, seed=77)
    batches = list(data.batches(pts))
    st, cn = build_gpu(sim, batches, (mn, mx))
    o = build_oracle(batches, (mn, mx))
    assert st.dbg == 0 and o.stats().droppedSpilledPoints == 0
    assert_same_octree(st, cn, o.stats(), o.canon(), "uniform 3x1M: ours vs oracle")
    assert o.check_voxel_colors(cn) == 0


def test_spill_buffer_overflow_postpones_splits_and_loses_nothing(sim):
    """64 level-2 leaves of a uniform stream cross 50 000 points in the same 100 k-point batch: 64 x ~49.2 k stored points
    exceed the 3 Mi-entry spill buffer (the reference re-inserts at most 3 000 001 spilled points per batch and silently
    drops the rest, voxels.cu:628 — a regime where it is not defined). Here the splits that do not fit are refused as a
    whole and requested again in the next batch: Stats::dbg bit 0 is raised, no point is lost, the octree stays valid."""
    n = 3_600_000
    pts, mn, mx = data.uniform_cube(n, size=1024.0, seed=123)
    sim.set_box(mn, mx)
    sim.reset()
    sim.insert_batches(list(data.batches(pts, 100_000)))
    st = sim.stats()
    assert st.numPointsProcessed == n and st.numPoints == n, (st.numPoints, st.dbg)
    assert st.dbg & 0x56 == 0                                   # nothing was dropped
    cn = oracle.canon_from_image(*sim.download_octree())         # raises if the image is inconsistent
    leaves = cn.records[cn.records["isLeaf"] == 1]
    assert int(leaves["numPoints"].sum()) == n and (leaves["numPoints"] <= 64_000).all()
    # with a stream that does not overflow, the same code path is the oracle's (regression guard for the refusal logic)
    if st.dbg & 1:
        assert (cn.records["level"] <= 4).all()


def test_shell_stream_vs_reference_kernels(sim):
    pts, mn, mx = data.shell(2_400_000)
    batches = list(data.batches(pts))
    st, cn = build_gpu(sim, batches, (mn, mx))
    assert_reference_octree(st, cn, "shell_stream", "shell: ours vs reference kernels")
