"""What the original project's own kernels and loaders produced, recorded once as golden data (tests/golden/
make_golden_reference.py, tests/golden/make_golden_loaders.py), and the digests both sides are reduced to.

The tests compare our results with these records, so they need neither the original sources nor its compiled kernels.
Octrees are stored in canonical form (DESIGN.md §3). A frame is stored as: the Stats::numVisible* counters, the
Node::visible / isLarge flags in canonical node order, a SHA-256 of the depth words of the u64 framebuffer, and a
SHA-256 of the whole framebuffer and of the surface. Which point donates a voxel's colour is a race (DESIGN.md §3), so a
frame coloured by its samples cannot be reproduced word for word from one build to the next; for those frames the whole
framebuffer and surface are taken from the same view re-drawn with colorByNode, whose colours depend on the node only.
"""
import hashlib
import os
import types

import numpy as np

import oracle

HERE = os.path.dirname(os.path.abspath(__file__))
KERNELS = os.path.join(HERE, "golden", "reference_parity_b200.npz")
LOADERS = os.path.join(HERE, "golden", "reference_loaders.npz")
ABI_LAYOUT = os.path.join(HERE, "golden", "reference_abi_layout.txt")
RGB_MASK = np.uint32(0x00FFFFFF)       # the original LAS loader leaves alpha uninitialised

_cache = {}


def _load(path):
    if path not in _cache:
        with np.load(path) as z:
            _cache[path] = dict(z)
    return _cache[path]


def kernels():
    return _load(KERNELS)


def loaders():
    return _load(LOADERS)


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def points_digest(p, with_color=True):
    cols = [p[a].view(np.uint32) for a in "xyz"]
    if with_color:
        cols.append(p["color"] & RGB_MASK)
    return sha(np.stack(cols, axis=1) if len(p) else np.zeros((0, len(cols)), np.uint32))


# ---- octrees ---------------------------------------------------------------------------------------------------

def octree_digest(stats, canon=None):
    d = {"stats": np.array([int(getattr(stats, f)) for f in oracle.STATS_FIELDS], dtype=np.uint64)}
    if canon is not None:
        d["records"] = canon.records
    return d


def octree(key):
    """The recorded octree `key` as an object compare_canon / compare_stats accept (records, stats)."""
    g = kernels()
    stats = types.SimpleNamespace(**{f: int(v) for f, v in zip(oracle.STATS_FIELDS, g[key + "/stats"])})
    return types.SimpleNamespace(records=g.get(key + "/records"), stats=stats)


# ---- frames ----------------------------------------------------------------------------------------------------

VISIBLE = ("numVisibleNodes", "numVisibleInner", "numVisibleLeaves", "numVisiblePoints", "numVisibleVoxels")


def frame_digest(sim, canon=None):
    """Digest of the frame the last sim.render() drew (see the module docstring). With `canon` (the canonical form of
    the octree on the device) the visibility flags are included, in canonical node order."""
    st = sim.stats()
    fb, su = sim.framebuffer(), sim.surface()
    d = {"visible": np.array([getattr(st, f) for f in VISIBLE], dtype=np.uint32),
         "depth": sha((fb >> np.uint64(32)).astype(np.uint32))}
    if canon is not None:
        nodes = sim.memcpy_dtoh(sim.buffers().nodes, st.numNodes * 152).reshape(-1, 152)
        d["flags"] = nodes[canon.records["nodeIndex"]][:, [116, 119]]
    if not (sim.uniforms.colorByNode or sim.uniforms.colorByLOD):
        sim.set_settings(colorByNode=1)
        sim.render()
        fb, su = sim.framebuffer(), sim.surface()
        sim.set_settings(colorByNode=0)
    d["framebuffer"] = sha(fb)
    d["surface"] = sha(su)
    return d


def frame_diffs(got, key, want=None):
    """Differences between a frame digest and the recorded one (or `want`), as readable lines."""
    if want is None:
        g = kernels()
        want = {k[len(key) + 1:]: v for k, v in g.items() if k.startswith(key + "/")}
    assert want, "no golden frame " + key
    diffs = []
    for k in ("visible", "flags", "depth", "framebuffer", "surface"):
        if k not in want:
            continue
        a, b = got[k], want[k]
        if a.shape != b.shape or not (a == b).all():
            detail = ""
            if k == "visible":
                detail = ": %s != %s" % (a.tolist(), b.tolist())
            elif k == "flags" and a.shape == b.shape:
                detail = ": %d flags differ" % int((a != b).sum())
            diffs.append("%s: %s differs%s" % (key, k, detail))
    return diffs
