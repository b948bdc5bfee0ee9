"""LAS front-end row (SURVEY.md §8f-2): record decode. CPU part pins the oracle against what the reference's
own LasLoader.cpp read from the same files (tests/golden/reference_loaders.npz); GPU part pins our device decode
against both."""
import numpy as np
import pytest

import oracle
import reference_golden as golden
from simlod_b200 import data

SCALE = (0.001, 0.002, 0.0005)
OFFSET = (10.0, -5.0, 2.5)
TRANSLATION = (-1.0, 3.0, 0.125)
RGB_MASK = golden.RGB_MASK             # the reference leaves alpha uninitialised (LasLoader.cpp:190-195)
RGB_FORMATS = (2, 3, 5, 7)
DECODE_POINTS = 60_000
DECODE_CASES = [(2, True, 0), (2, False, 0), (3, True, 0), (0, True, 0), (1, True, 0),
                (5, True, 0), (7, True, 0), (2, True, 1), (3, False, 3)]      # 5: 63-byte records; odd extra bytes
DECODE_WINDOWS = ((0, 60_000), (123, 4_567), (59_999, 1))
DEVICE_POINTS = 700_001
DEVICE_CASES = [(2, 0), (3, 0), (0, 0), (5, 0), (7, 0), (2, 1), (0, 3)]      # odd record sizes: every other record on an odd address
DEVICE_SIZES = [300_000, 255, 0, 400_001 - 255]                                # full tiles, a ragged tile, an empty batch


def decode_key(fmt, wide, extra, first, count):
    """Golden key of the reference's decode of records first..first+count of a file written with these settings."""
    return "las/%d_%d_%d/%d_%d" % (fmt, int(wide), extra, first, count)


def assert_same_as_reference(points, fmt, wide, extra, first, count):
    want = golden.loaders()[decode_key(fmt, wide, extra, first, count)]
    assert (golden.points_digest(points, with_color=fmt in RGB_FORMATS) == want).all(), (fmt, wide, extra, first, count)


def same_points(a, b, with_color=True):
    ok = all((a[ax].view(np.uint32) == b[ax].view(np.uint32)).all() for ax in "xyz")
    if with_color:
        ok = ok and ((a["color"] & RGB_MASK) == (b["color"] & RGB_MASK)).all()
    return bool(ok)


@pytest.mark.parametrize("fmt,wide,extra", DECODE_CASES)
def test_oracle_decode_matches_reference_lasloader(tmp_path, fmt, wide, extra):
    pts, _, _ = data.terrain(DECODE_POINTS)
    path = str(tmp_path / "t.las")
    rec = data.write_las(path, pts, fmt=fmt, scale=SCALE, offset=OFFSET, wide_colors=wide, extra_bytes=extra)
    hdr = 227          # the records follow the header in the file the reference read
    assert (np.fromfile(path, dtype=np.uint8)[hdr:].reshape(rec.shape) == rec).all()
    for first, count in DECODE_WINDOWS:
        got = oracle.decode_las(rec[first:first + count], count, rec.shape[1], fmt, SCALE, OFFSET, TRANSLATION)
        assert_same_as_reference(got, fmt, wide, extra, first, count)


def test_decode_roundtrip_properties():
    # decode(encode(p)) is within half a quantum of p, and 16-bit colours come back as the 8-bit originals
    pts, _, _ = data.terrain(20_000)
    for fmt in (2, 3):
        rec = data.las_records(pts, fmt, SCALE, OFFSET)
        got = oracle.decode_las(rec, len(pts), rec.shape[1], fmt, SCALE, OFFSET)
        for k, ax in enumerate("xyz"):
            assert np.abs(got[ax].astype(np.float64) - pts[ax].astype(np.float64)).max() <= SCALE[k] * 0.5 + 1e-4
        assert ((got["color"] & RGB_MASK) == (pts["color"] & RGB_MASK)).all()
    empty = oracle.decode_las(np.zeros(0, np.uint8), 0, 26, 2, SCALE, OFFSET)
    assert len(empty) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,extra", DEVICE_CASES)
def test_device_decode_matches_oracle_and_reference(tmp_path, fmt, extra):
    from simlod_b200 import SimLOD
    pts, mn, mx = data.terrain(DEVICE_POINTS)
    path = str(tmp_path / "t.las")
    rec = data.write_las(path, pts, fmt=fmt, scale=SCALE, offset=OFFSET, extra_bytes=extra)
    sim = SimLOD(320, 176, persistent_bytes=2 << 30)
    try:
        sim.set_box(mn, mx)
        sim.reset()
        layout = sim.las_layout(rec.shape[1], fmt, SCALE, OFFSET, TRANSLATION)
        first = 0
        for slot, n in enumerate(DEVICE_SIZES):
            sim.upload_batch_las(rec[first:first + n], n, layout)
            got = sim.ring_slot(slot, n)
            want = oracle.decode_las(rec[first:first + n], n, rec.shape[1], fmt, SCALE, OFFSET, TRANSLATION)
            assert same_points(got, want, with_color=True), (fmt, slot)
            if n:
                assert_same_as_reference(got, fmt, True, extra, first, n)
            first += n
    finally:
        sim.close()


@pytest.mark.gpu
def test_las_stream_builds_the_same_octree_as_decoded_points():
    from simlod_b200 import SimLOD
    pts, mn, mx = data.terrain(1_500_000)
    rec = data.las_records(pts, 2, SCALE, (0.0, 0.0, 0.0))
    dec = oracle.decode_las(rec, len(pts), rec.shape[1], 2, SCALE, (0.0, 0.0, 0.0))
    sim = SimLOD(320, 176, persistent_bytes=3 << 30)
    try:
        sim.set_box(mn, mx)
        layout = sim.las_layout(rec.shape[1], 2, SCALE, (0.0, 0.0, 0.0))
        sim.reset()
        for s in range(0, len(pts), 1_000_000):
            n = min(1_000_000, len(pts) - s)
            sim.upload_batch_las(rec[s:s + n], n, layout)
            while sim.update_octree() is not None and sim.stats().batchletIndex < s // 1_000_000 + 1:
                pass
        st_a = sim.stats()
        cn_a = oracle.canon_from_image(*sim.download_octree())
        sim.reset()
        sim.insert_batches(data.batches(dec))
        st_b = sim.stats()
        cn_b = oracle.canon_from_image(*sim.download_octree())
        assert not oracle.compare_canon(cn_a, cn_b) and not oracle.compare_stats(st_a, st_b)
        # (alpha differs by construction: device decode writes 0xff, hashes include it, so dec carries 0xff too)
    finally:
        sim.close()
