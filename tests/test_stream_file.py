"""Streaming front-end row (SURVEY.md §8f-1): .simlod container, what the reference's own loader read from it
(tests/golden/reference_loaders.npz) as CPU reference, and (GPU) the file streamer: header -> box, reset, loader
threads + pinned pool + in-order upload."""
import os

import numpy as np
import pytest

import oracle
import reference_golden as golden
from simlod_b200 import data

SIMLOD_POINTS = 123_457
SIMLOD_WINDOWS = ((0, 123_457), (100_000, 23_457), (5, 1))


def test_simlod_container_roundtrip_through_reference_loader(tmp_path):
    pts, mn, mx = data.terrain(SIMLOD_POINTS)
    path = str(tmp_path / "t.simlod")
    data.write_simlod(path, pts, mn, mx)
    assert os.path.getsize(path) == 24 + 16 * len(pts)
    hdr = np.fromfile(path, dtype="<f4", count=6)
    assert np.allclose(hdr[:3], mn) and np.allclose(hdr[3:], mx)
    for first, count in SIMLOD_WINDOWS:
        # loadFileNative (SimlodLoader.cpp:147-157) reads count * 16 bytes at 24 + first * 16
        got = np.fromfile(path, dtype=oracle.POINT_DTYPE, count=count, offset=24 + first * 16)
        assert (got == pts[first:first + count]).all()
        assert (golden.sha(got) == golden.loaders()["simlod/%d_%d" % (first, count)]).all(), (first, count)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 6])
def test_file_streamer_builds_the_same_octree_as_in_memory_batches(tmp_path, threads):
    from simlod_b200 import SimLOD
    n = 3_300_123
    pts, mn, mx = data.terrain(n)
    path = str(tmp_path / "scan.simlod")
    data.write_simlod(path, pts, mn, mx)
    sim = SimLOD(320, 176, persistent_bytes=3 << 30)
    try:
        got_n, kms, tms = sim.insert_simlod_file(path, loader_threads=threads)
        assert got_n == n and kms > 0 and tms >= kms * 0.5
        st_a = sim.stats()
        assert st_a.numPointsProcessed == n and st_a.batchletIndex == 4 and st_a.dbg == 0
        assert [sim.uniforms.boxMax[i] for i in range(3)] == [np.float32(mx[i] - mn[i]) for i in range(3)]
        cn_a = oracle.canon_from_image(*sim.download_octree())
        sim.set_box(mn, mx)
        sim.reset()
        sim.insert_batches(data.batches(pts))
        st_b = sim.stats()
        cn_b = oracle.canon_from_image(*sim.download_octree())
        assert not oracle.compare_canon(cn_a, cn_b) and not oracle.compare_stats(st_a, st_b)
    finally:
        sim.close()


@pytest.mark.gpu
def test_file_streamer_unbuffered_reads_build_the_same_octree(tmp_path):
    """SIMLOD_STREAM_DIRECT (O_DIRECT block reads, the cold-file path): same octree as the buffered path, for a file whose
    pages were dropped from the page cache. Skipped where the file system cannot do O_DIRECT (tmpfs)."""
    from simlod_b200 import SimLOD, SimlodError
    n = 2_100_007                                  # ends in the middle of a 4 KB block
    pts, mn, mx = data.terrain(n)
    path = str(tmp_path / "cold.simlod")
    data.write_simlod(path, pts, mn, mx)
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
        os.posix_fadvise(fd, 0, 0, os.POSIX_FADV_DONTNEED)       # evict the (clean) pages: the next read comes from the device
    finally:
        os.close(fd)
    sim = SimLOD(320, 176, persistent_bytes=3 << 30)
    try:
        try:
            got_n, kms, tms = sim.insert_simlod_file(path, loader_threads=5, direct=True)
        except SimlodError as e:
            if "O_DIRECT" in str(e):
                pytest.skip("file system of %s does not support O_DIRECT" % tmp_path)
            raise
        st_a = sim.stats()
        assert got_n == n and st_a.numPoints == n and st_a.dbg == 0
        cn_a = oracle.canon_from_image(*sim.download_octree())
        sim.insert_simlod_file(path, loader_threads=5)
        st_b = sim.stats()
        cn_b = oracle.canon_from_image(*sim.download_octree())
        assert not oracle.compare_canon(cn_a, cn_b) and not oracle.compare_stats(st_a, st_b)
    finally:
        sim.close()


@pytest.mark.gpu
def test_file_streamer_rejects_bad_input(tmp_path):
    from simlod_b200 import SimLOD, SimlodError
    sim = SimLOD(320, 176, persistent_bytes=1 << 30)
    try:
        with pytest.raises(SimlodError):
            sim.insert_simlod_file(str(tmp_path / "missing.simlod"))
        p = tmp_path / "short.simlod"
        p.write_bytes(b"1234")
        with pytest.raises(SimlodError):
            sim.insert_simlod_file(str(p))
        # header only: an empty scan is fine
        data.write_simlod(str(tmp_path / "empty.simlod"), np.zeros(0, dtype=oracle.POINT_DTYPE), (0, 0, 0), (1, 1, 1))
        n, _, _ = sim.insert_simlod_file(str(tmp_path / "empty.simlod"))
        assert n == 0 and sim.stats().numPoints == 0
    finally:
        sim.close()
