"""Records tests/golden/reference_parity_b200.npz on a B200 by running the UNMODIFIED reference kernels
(oracle/_ref/*.cubin, compiled by oracle/build_ref.cpp from the original project's sources) through the headless
launch surface, on the inputs of tests/test_parity_gpu.py and tests/test_full_size_gpu.py:

    python tests/golden/make_golden_reference.py OUT.npz

Octrees are built by the reference's kernel_construct / kernel (reset); frames are drawn by the reference's
kernel_render on the octree OUR builder made, exactly as the tests then draw it with ours. Every record is also checked
against ours live, here, so a recording is only written when both agree; the tests then compare with the recording
(tests/reference_golden.py says what a frame digest holds)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)

import oracle  # noqa: E402
import reference_golden as golden  # noqa: E402
import test_full_size_gpu as tf  # noqa: E402
import test_parity_gpu as tp  # noqa: E402
from simlod_b200 import SimLOD, camera, data  # noqa: E402

OUT = {}


def use_reference(sim, programs, on):
    for p in programs:
        sim.use_module(p, oracle.REF_CUBINS[p] if on else None)


def put(key, digest):
    for k, v in digest.items():
        OUT[key + "/" + k] = v


def octree_case(sim, key, batches, box, rcp_check=None):
    """Reference octree of `batches`, checked against ours; stores records + stats."""
    st, cn = tp.build_gpu(sim, batches, box)
    use_reference(sim, (0, 2), True)
    st_r, cn_r = tp.build_gpu(sim, batches, box)
    use_reference(sim, (0, 2), False)
    tp.assert_same_octree(st, cn, st_r, cn_r, key + ": ours vs reference kernels")
    put(key, golden.octree_digest(st_r, cn_r))
    return st_r, cn_r


def frame_case(sim, key, canon=None):
    """The current view drawn by ours and by the reference's kernel_render; both digests must agree."""
    sim.render()
    ours = golden.frame_digest(sim, canon)
    use_reference(sim, (1,), True)
    sim.render()
    ref = golden.frame_digest(sim, canon)
    use_reference(sim, (1,), False)
    diffs = golden.frame_diffs(ours, key, ref)
    assert not diffs, "\n".join(diffs)
    put(key, ref)


def parity(sim):
    pts, mn, mx = data.uniform_cube(1_000_000)
    st_r, cn_r = octree_case(sim, "config1_uniform_1m", [pts], (mn, mx))
    assert tp.build_oracle([pts], (mn, mx)).check_voxel_colors(cn_r) == 0
    batches, box = tp.terrain_batches()
    octree_case(sim, "streamed_ragged_terrain", batches, box)
    pts, mn, mx = data.uniform_cube(120_000, size=64.0, seed=5)
    octree_case(sim, "small_batches", tp.split(pts, [20_000, 20_000, 10_000, 1, 30_000, 39_999]), (mn, mx))
    pts, mn, mx = data.shell(2_400_000)
    octree_case(sim, "shell_stream", list(data.batches(pts)), (mn, mx))

    for dataset in ("uniform", "terrain"):
        for hqs in (0, 1):
            if dataset == "uniform":
                pts, mn, mx = data.uniform_cube(1_000_000)
                batches = [pts]
            else:
                pts, mn, mx = data.terrain(4_000_000)
                batches = list(data.batches(pts))
            _, cn = tp.build_gpu(sim, batches, (mn, mx))
            sim.set_settings(useHighQualityShading=hqs, pointSize=1)
            for name, (view, proj) in tp.cameras(mx, sim.width, sim.height):
                sim.set_camera(view, proj)
                frame_case(sim, "framebuffer/%s/hqs%d/%s" % (dataset, hqs, name), cn)
            sim.set_settings(useHighQualityShading=0)

    pts, mn, mx = data.terrain(2_000_000)
    _, cn = tp.build_gpu(sim, list(data.batches(pts)), (mn, mx))
    view, proj = camera.autofocus(mx, sim.width, sim.height)
    sim.set_camera(view, proj)
    for k, settings in enumerate(tp.LOD_COLOUR_SETTINGS):
        sim.set_settings(pointSize=1, colorByLOD=0, colorByNode=0, useHighQualityShading=0)
        sim.set_settings(**settings)
        frame_case(sim, "lod_colours/%d" % k, cn)
    sim.set_settings(pointSize=1, colorByLOD=0, colorByNode=0, useHighQualityShading=0)

    pts, mn, mx = data.terrain(2_000_000)
    _, cn = tp.build_gpu(sim, list(data.batches(pts)), (mn, mx))
    r = float(np.linalg.norm(mx))
    far = camera.orbit_camera(-2.0, -0.9, r * 6.0, (mx[0] * 0.5, mx[1] * 0.5, 0.0), sim.width, sim.height)
    close = camera.orbit_camera(0.4, -0.3, r * 0.08, (mx[0] * 0.55, mx[1] * 0.45, mx[2] * 0.3), sim.width, sim.height)
    for hqs in (0, 1):
        sim.set_settings(useHighQualityShading=hqs)
        sim.set_camera(*far)
        sim.set_camera(*close, update_visibility=False)
        frame_case(sim, "frozen/hqs%d/frozen" % hqs, cn)
        sim.set_camera(*close)
        frame_case(sim, "frozen/hqs%d/moved" % hqs, cn)
    sim.set_settings(useHighQualityShading=0)

    # the chunk-list cache sequence; the reference's own renders are the "other kernel" that scribbles over the buffer
    pts, mn, mx = data.terrain(5_000_000)
    batches = list(data.batches(pts))
    sim.set_settings(pointSize=1, colorByLOD=0, colorByNode=0, useHighQualityShading=0)
    view, proj = camera.autofocus(mx, sim.width, sim.height)
    sim.set_camera(view, proj)
    tp.build_gpu(sim, batches[:3], (mn, mx))
    frame_case(sim, "chunk_cache/first frame")
    sim.render(); sim.render()
    frame_case(sim, "chunk_cache/after another kernel used the buffer")
    for b in batches[3:]:
        sim.upload_batch(b)
    while sim.stats().batchletIndex < len(batches):
        sim.update_octree()
    sim.render(); sim.render()
    frame_case(sim, "chunk_cache/after growth")
    other, _, _ = data.terrain(3_000_000, seed=11)
    sim.render()
    tp.build_gpu(sim, list(data.batches(other)), (mn, mx))
    frame_case(sim, "chunk_cache/after a reset")
    sim.set_settings(useHighQualityShading=1)
    sim.render()
    frame_case(sim, "chunk_cache/hqs")
    sim.set_settings(useHighQualityShading=0)


def full_size():
    n = 36 * tf.BATCH
    sim = SimLOD(1920, 1080, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=6 << 30, render_blocks_per_sm=3)
    try:
        dptr = sim.device_alloc(n * 16)
        sim.generate(sim.GEN_TERRAIN, dptr, n, 0, n, 7)
        box = ((0.0, 0.0, 0.0), data.TERRAIN_EXTENT)
        st = tf.build(sim, dptr, n, box)
        cn = oracle.canon_from_image(*sim.download_octree())
        use_reference(sim, (0, 2), True)
        st_r = tf.build(sim, dptr, n, box)
        use_reference(sim, (0, 2), False)
        cn_r = oracle.canon_from_image(*sim.download_octree())
        tp.assert_same_octree(st, cn, st_r, cn_r, "36M: ours vs reference kernels")
        put("config2_36m", golden.octree_digest(st_r, cn_r))
    finally:
        sim.close()

    n = 350 * tf.BATCH
    sim = SimLOD(1920, 1080, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=24 << 30, render_blocks_per_sm=3)
    try:
        dptr = sim.device_alloc(n * 16)
        sim.generate(sim.GEN_TERRAIN, dptr, n, 0, n, 7)
        box = ((0.0, 0.0, 0.0), data.TERRAIN_EXTENT)
        use_reference(sim, (0, 2), True)
        st_r = tf.build(sim, dptr, n, box)
        use_reference(sim, (0, 2), False)
        st = tf.build(sim, dptr, n, box)
        tp.assert_same_octree(st, types_canon(), st_r, types_canon(), "350M: ours vs reference kernels")
        put("config3_350m", golden.octree_digest(st_r))
        for hqs in (0, 1):
            sim.set_settings(useHighQualityShading=hqs, pointSize=1)
            for k, (view, proj) in enumerate(tf.cameras(data.TERRAIN_EXTENT, sim.width, sim.height)):
                sim.set_camera(view, proj)
                frame_case(sim, "config5/hqs%d/camera%d" % (hqs, k))
        sim.set_settings(useHighQualityShading=0)
    finally:
        sim.close()

    n = 250 * tf.BATCH
    sim = SimLOD(640, 360, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=24 << 30)
    try:
        dptr = sim.device_alloc(n * 16)
        sim.generate(sim.GEN_SHELL, dptr, n, 0, n, 1234)
        box = ((0.0, 0.0, 0.0), (data.SHELL_CUBE,) * 3)
        use_reference(sim, (0, 2), True)
        st_r = tf.build(sim, dptr, n, box)
        use_reference(sim, (0, 2), False)
        st = tf.build(sim, dptr, n, box)
        tp.assert_same_octree(st, types_canon(), st_r, types_canon(), "config 4: ours vs reference kernels")
        put("config4_shell_250m", golden.octree_digest(st_r))
    finally:
        sim.close()


def types_canon():
    """An empty canonical form: compares equal to another, so that only Stats are compared."""
    import types
    return types.SimpleNamespace(records=np.zeros(0, dtype=oracle.RECORD_DTYPE))


def main(out):
    assert all(os.path.exists(p) for p in oracle.REF_CUBINS.values()), "oracle/_ref/*.cubin not built"
    sim = SimLOD(1920, 1080, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=12 << 30, render_blocks_per_sm=3)
    try:
        parity(sim)
    finally:
        sim.close()
    full_size()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    np.savez_compressed(out, **OUT)
    print("wrote", out, len(OUT), "arrays,", os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else golden.KERNELS)
