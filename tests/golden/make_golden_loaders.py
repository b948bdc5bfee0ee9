"""Records, on the CPU, what the original project's own host code gives for the inputs of the loader and ABI tests:

    python tests/golden/make_golden_loaders.py REFERENCE_TREE

  tests/golden/reference_loaders.npz      digests of what loadLasNative (LasLoader.cpp) and loadFileNative
                                          (SimlodLoader.cpp), compiled into oracle/_ref/ by build(), read from the
                                          files tests/test_las.py and tests/test_stream_file.py write
  tests/golden/reference_abi_layout.txt   tests/native/abi_layout.cu built against the original headers
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path.insert(0, ROOT)
sys.path.insert(0, TESTS)

import oracle  # noqa: E402
import reference_golden as golden  # noqa: E402
import test_las as tl  # noqa: E402
import test_stream_file as ts  # noqa: E402
from simlod_b200 import build, data  # noqa: E402


def loaders(tmp):
    assert oracle.ref_las() is not None and oracle.ref_simlod() is not None, "oracle/_ref/ loaders not built"
    out = {}
    pts, _, _ = data.terrain(tl.DECODE_POINTS)
    path = os.path.join(tmp, "t.las")
    for fmt, wide, extra in tl.DECODE_CASES:
        data.write_las(path, pts, fmt=fmt, scale=tl.SCALE, offset=tl.OFFSET, wide_colors=wide, extra_bytes=extra)
        for first, count in tl.DECODE_WINDOWS:
            ref = oracle.ref_las_load(path, first, count, tl.TRANSLATION)
            out[tl.decode_key(fmt, wide, extra, first, count)] = golden.points_digest(ref, with_color=fmt in tl.RGB_FORMATS)
    pts, _, _ = data.terrain(tl.DEVICE_POINTS)
    for fmt, extra in tl.DEVICE_CASES:
        data.write_las(path, pts, fmt=fmt, scale=tl.SCALE, offset=tl.OFFSET, extra_bytes=extra)
        first = 0
        for n in tl.DEVICE_SIZES:
            if n:
                ref = oracle.ref_las_load(path, first, n, tl.TRANSLATION)
                out[tl.decode_key(fmt, True, extra, first, n)] = golden.points_digest(ref, with_color=fmt in tl.RGB_FORMATS)
            first += n
    pts, mn, mx = data.terrain(ts.SIMLOD_POINTS)
    path = os.path.join(tmp, "t.simlod")
    data.write_simlod(path, pts, mn, mx)
    for first, count in ts.SIMLOD_WINDOWS:
        out["simlod/%d_%d" % (first, count)] = golden.sha(oracle.ref_simlod_load(path, first, count))
    np.savez_compressed(golden.LOADERS, **out)
    print("wrote", golden.LOADERS, len(out), "digests")


def abi_layout(reference_tree, tmp):
    po = os.path.join(reference_tree, "modules", "progressive_octree")
    exe = os.path.join(tmp, "abi_layout_ref")
    subprocess.check_call([build.NVCC, "-std=c++17", "-DREFERENCE_HEADERS", "-I" + po, "-o", exe,
                           os.path.join(TESTS, "native", "abi_layout.cu")])
    text = subprocess.check_output([exe], text=True)
    with open(golden.ABI_LAYOUT, "w") as f:
        f.write(text)
    print("wrote", golden.ABI_LAYOUT, len(text.splitlines()), "lines")


if __name__ == "__main__":
    with tempfile.TemporaryDirectory() as tmp:
        loaders(tmp)
        abi_layout(sys.argv[1], tmp)
