"""Generates tests/golden/reference_kernels_b200.npz on a B200 by running the UNMODIFIED
reference kernels (oracle/_ref/*.cubin = the original sources compiled by oracle/build_ref.cpp
with the reference's own NVRTC/nvJitLink recipe) through the headless launch surface:

    python tests/golden/make_golden.py OUT.npz

For every case of tests/make_golden_cases.py it stores the canonical octree records, the
deterministic Stats fields, MUFU.RCP(cube size) and the packed u64 framebuffer of one frame, all
produced by the reference's kernel_construct / kernel / kernel_render. The CPU suite pins
oracle/oracle.cpp (builder, canonicaliser and rasteriser) to these; the GPU suite compares ours with
the recordings of tests/golden/make_golden_reference.py."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import make_golden_cases as cases  # noqa: E402
import oracle  # noqa: E402
from simlod_b200 import SimLOD  # noqa: E402


def main(out):
    sim = SimLOD(cases.GOLDEN_W, cases.GOLDEN_H, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=4 << 30)
    for p in (0, 1, 2):
        sim.use_module(p, oracle.REF_CUBINS[p])
    g = {}
    for name, batches, (mn, mx), (view, proj) in cases.cases():
        sim.set_box(mn, mx)
        sim.reset()
        sim.insert_batches(batches)
        st = sim.stats()
        cn = oracle.canon_from_image(*sim.download_octree())
        g[name + "/records"] = cn.records
        g[name + "/stats"] = np.array([int(getattr(st, f)) for f in oracle.STATS_FIELDS], dtype=np.uint64)
        size = max(b - a for a, b in zip(mn, mx))
        g[name + "/rcp"] = np.float32(sim.device_rcp(size))
        sim.set_camera(view, proj)
        sim.render()
        g[name + "/framebuffer"] = sim.framebuffer()
        s2 = sim.stats()
        g[name + "/visible"] = np.array([s2.numVisibleNodes, s2.numVisibleInner, s2.numVisibleLeaves, s2.numVisiblePoints, s2.numVisibleVoxels], dtype=np.uint32)
        g[name + "/uniforms"] = np.frombuffer(sim.uniforms_bytes(), dtype=np.uint8)
        print(name, "nodes", st.numNodes, "points", st.numPoints, "voxels", st.numVoxels, "visible", g[name + "/visible"])
    np.savez_compressed(out, **g)
    print("wrote", out)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_kernels_b200.npz"))
