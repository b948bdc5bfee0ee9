#!/usr/bin/env python
"""bench.py — octree insertion throughput (and render rate) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our sm_100a path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores (oracle port)

A step is one pass of the hot path over one batch: 1 000 000 synthetic XYZRGBA points (16 B each) inserted into the
growing octree by kernel_construct. The stream is BASELINE.json configs[2], the 350 M-point scan (Morro-Bay stand-in
terrain, generated), inserted from a freshly reset octree in spatially coherent 1 M-point batches. A timed PASS inserts
the first K = --steps batches of that stream (all 350 with --steps 350), the reported time is the median of >= 5 passes
from reset (SURVEY.md §8d), and ms_per_step is that time per 1 M-point batch; --warmup batches are inserted untimed
first. --dump-outputs DIR writes the octree the last timed pass built (canonical form, DESIGN.md §3) as .npy files.

With N > 1 every rank owns a complete builder and inserts its own 350 M-point scan tile of the same extent and density
(tile g of a survey of N tiles): per-GPU work is identical to N = 1, scaling is weak, and there is no data-path
collective (NCCL carries barrier / max-time / stats reductions only). BASELINE.json configs[3] as SURVEY.md §8d defines
it — ONE sphere shell of N x 250 M points, rank g inserts the batches b = g (mod N) — is measured next to it and reported
under `config4`; ONE octree over the N GPUs (spatial exchange over NVLink peer memory, SURVEY.md §8f-3) under
`merged_octree`.

Numbers:
  value        Mpoints/s, all ranks' points / max-over-ranks median device time of a pass, batches already resident
               in HBM and consumed in place (simlod_insert_device maps the 50-slot ring window onto the caller's buffer;
               all launch gaps are inside the timed region)
  e2e          same metric through the public API from pinned HOST memory: per step one 16 MB host->device copy
               and one 112-byte Stats read-back per launch inside the timed region
  roofline     kernel_construct: algorithmic bytes (16 in + 16 out + 32*s + 16*v per point, SURVEY.md §8d)
               / summed launch time (CUDA events on the launch stream) against the measured HBM copy peak
  reference_gpu  the UNMODIFIED reference kernels (oracle/_ref/*.cubin, compiled from /root/reference by
               oracle/build_ref.cpp) through simlod_use_module on the same GPU, same buffers, same input, with their
               native grids (1 block/SM construct, occupancy render): the numbers to beat (SURVEY.md §8d-i)
  render       kernel_render on the built octree, 6 cameras x {atomicMin, HQS}, with the per-frame HBM roofline
               (16 B/sample + 12*W*H, HQS 32 B/sample + 28*W*H) and the reference kernel beside it
  cpu_baseline the CPU oracle (port of the reference algorithm, 1 thread) on a bounded sample
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 1_000_000
METRIC = "Mpoints/sec octree insertion (16B XYZRGBA)"
CONFIG3_BATCHES = 350            # BASELINE.json configs[2]: 350 M points
CONFIG4_BATCHES_PER_GPU = 250    # BASELINE.json configs[3]: 250 M points per GPU of one N x 250 M shell
TERRAIN_SEED, SHELL_SEED = 7, 1234
W_PX, H_PX = 1920, 1080


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--passes", type=int, default=5, help="timed passes over the whole stream (median reported)")
    ap.add_argument("--batches", type=int, default=CONFIG3_BATCHES, help="developer knob: batches of the stream (350 = config 3)")
    ap.add_argument("--cpu-sample-batches", type=int, default=16, help="batches of the stream the 1-thread CPU oracle inserts for cpu_baseline (about 6-10 s)")
    ap.add_argument("--no-render", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the LAS / file-streamer / config-4 legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the octree of the last timed pass to DIR/*.npy")
    return ap.parse_args()


def workload_name(batches):
    return "terrain_synth_%dM (Morro Bay %dM stand-in: 4800x4300x300 m fBm terrain in 50 m flight strips), %d x 1M-point batches per GPU streamed from a reset octree" % (
        batches, batches, batches)


# ---- clocks sampled DURING the timed regions (B200_PROFILING.md) --------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.rows = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, windows):
        sm, mx, reasons = [], 0, set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7 or not any(a <= t <= b + 0.15 for a, b in windows):
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:      # timed regions shorter than the sampling period: fall back to all samples
            for t, line in self.rows:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0])); mx = max(mx, float(f[1]))
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def recorded_traffic(batches):
    """DRAM bytes per kernel_construct launch of THIS workload from the committed ncu launch list, if one exists
    (profiles/r02/ncu_construct_traffic_<batches>M.json, written by tools/ncu_traffic.py)."""
    p = os.path.join(ROOT, "profiles", "r02", "ncu_construct_traffic_%dM.json" % batches)
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def cameras(box_max):
    from simlod_b200 import camera
    cams = [("autofocus+%d" % k, camera.autofocus(box_max, W_PX, H_PX, yaw_offset=k * np.pi / 2)) for k in range(4)]
    cams += [("morro_bird", camera.orbit_camera(width=W_PX, height=H_PX, **camera.MORRO_BIRD)),
             ("morro_close", camera.orbit_camera(width=W_PX, height=H_PX, **camera.MORRO_CLOSE))]
    return cams


def render_sweep(sim, box_max, peak):
    """6 cameras x {atomicMin path, HQS}: best of 3 frames each, with the frame's algorithmic HBM bytes against the peak."""
    out = {}
    for hqs in (0, 1):
        sim.set_settings(useHighQualityShading=hqs)
        frames = []
        for name, (view, proj) in cameras(box_max):
            sim.set_camera(view, proj)
            sim.render()
            ms = min(sim.render() for _ in range(3))
            s = sim.stats()
            samples = s.numVisiblePoints + s.numVisibleVoxels
            alg = (32 * samples + 28 * W_PX * H_PX) if hqs else (16 * samples + 12 * W_PX * H_PX)
            gbs = alg / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            frames.append({"camera": name, "ms": round(ms, 4), "visible_nodes": s.numVisibleNodes, "samples": samples,
                           "msamples_per_s": round(samples / ms / 1e3, 1) if ms > 0 else None,
                           "roofline": {"achieved": round(gbs, 1), "frac": round(gbs / peak, 4)}})
        tot_samples = sum(f["samples"] for f in frames)
        tot_ms = sum(f["ms"] for f in frames)
        tot_alg = sum((32 if hqs else 16) * f["samples"] + (28 if hqs else 12) * W_PX * H_PX for f in frames)
        out["hqs" if hqs else "atomic_min"] = {
            "msamples_per_s": round(tot_samples / tot_ms / 1e3, 1), "fps": round(1e3 * len(frames) / tot_ms, 1),
            "roofline": {"bound": "hbm", "achieved": round(tot_alg / (tot_ms * 1e-3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(tot_alg / (tot_ms * 1e-3) / 1e9 / peak, 4),
                         "min_frac": min(f["roofline"]["frac"] for f in frames)},
            "frames": frames}
    sim.set_settings(useHighQualityShading=0)
    return out


def timed_passes(sim, insert, n_points, passes, barrier, windows):
    """`passes` x (reset, L2 flush, insert the whole stream): returns the per-pass (kernel_ms, total_ms) lists."""
    ks, ts = [], []
    for _ in range(passes):
        sim.reset()
        sim.flush_l2()
        barrier()
        t0 = time.time()
        kms, tms = insert()
        barrier()
        windows.append((t0, time.time()))
        ks.append(kms); ts.append(tms)
        st = sim.stats()
        assert st.numPointsProcessed == n_points and st.numPoints == n_points and st.dbg & 0x56 == 0, (st.numPointsProcessed, st.numPoints, st.dbg)
    return ks, ts


def bench_reference_gpu(device, dptr, n_batches, box, peak, ours_octree_sim):
    """The reference's own kernels on this GPU (SURVEY.md §8d-i): insertion of the same stream through the same harness
    with the reference launch shape (1 block per SM, main.cpp:370-371), and kernel_render on the SAME octree our
    rasteriser was timed on (ref_render.cubin swapped in, its occupancy grid)."""
    import oracle
    from simlod_b200 import SimLOD
    out = {"kernels": "oracle/_ref/ref_{construct,render,reset}.cubin = the unmodified /root/reference sources, NVRTC + nvJitLink as CudaModularProgram.h:84-98,214-239, sm_100"}
    if not all(os.path.exists(p) for p in oracle.REF_CUBINS.values()):
        out["unavailable"] = "oracle/_ref/*.cubin not built"
        return out
    npts = n_batches * BATCH
    # render first: on the octree our kernels built (frames were shown bit-identical by the parity suite)
    try:
        ours_octree_sim.use_module(1, oracle.REF_CUBINS[1])
        out["render_blocks"] = ours_octree_sim.launch_info()["render_blocks"]
        out["render"] = render_sweep(ours_octree_sim, box[1], peak)
    except Exception as e:
        out["render_error"] = repr(e)
    finally:
        ours_octree_sim.use_module(1, None)
    sim = None
    # the reference's reset kernel printf's "resetting octree" from the device: keep that off this process's stdout
    # (one JSON line is the contract) by pointing fd 1 at /dev/null while its kernels run
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        sim = SimLOD(W_PX, H_PX, device=device, momentary_bytes=oracle.REF_MOMENTARY_BYTES, persistent_bytes=max(8 << 30, n_batches * (96 << 20)),
                     construct_blocks_per_sm=1)
        for p in (0, 2):
            sim.use_module(p, oracle.REF_CUBINS[p])
        sim.set_box(*box)
        sim.reset(grid=(1, 1)); sim.insert_device(dptr, 3 * BATCH)
        ks, ts = [], []
        for _ in range(2):
            sim.reset(grid=(1, 1)); sim.flush_l2()
            kms, tms = sim.insert_device(dptr, npts)
            st = sim.stats()
            assert st.numPoints == npts, (st.numPoints, st.numPointsProcessed)
            ks.append(kms); ts.append(tms)
        out.update({"insert_kernel_ms": round(min(ks), 3), "insert_mpoints_per_s": round(npts / min(ks) / 1e3, 1),
                    "insert_total_mpoints_per_s": round(npts / min(ts) / 1e3, 1),
                    "construct_blocks": sim.launch_info()["construct_blocks"], "passes": 2,
                    "octree": {"numNodes": st.numNodes, "numVoxels": st.numVoxels}})
    except Exception as e:
        out["insert_error"] = repr(e)
    finally:
        if sim is not None:
            try:
                sim.synchronize()
            except Exception:
                pass
            sim.close()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout); os.close(devnull)
    return out


def bench_las(sim_device, host_batches, mn, mx):
    """LAS format-2 records (26 B/point) -> 16-byte points: device decode with the records resident in HBM, end to end
    from pinned host memory, and the reference's own CPU loader (oracle/_ref/libref_las.so = LasLoader.cpp) beside it."""
    import tempfile
    import oracle
    from simlod_b200 import SimLOD, data
    nb = len(host_batches)
    scale, offset = (0.001, 0.001, 0.001), (0.0, 0.0, 0.0)
    recs = [data.las_records(b, 2, scale, offset) for b in host_batches]
    bpp = recs[0].shape[1]
    n = nb * BATCH
    sim = SimLOD(320, 176, device=sim_device, persistent_bytes=1 << 30)
    out = {"format": 2, "bytes_per_point": bpp, "points": n}
    try:
        sim.set_box(mn, mx)
        layout = sim.las_layout(bpp, 2, scale, offset)
        dptr = sim.device_alloc(n * bpp)
        hptr = sim.host_alloc(n * bpp)
        host = np.ctypeslib.as_array((ctypes.c_uint8 * (n * bpp)).from_address(hptr))
        host[:] = np.concatenate(recs).reshape(-1)
        sim.memcpy_htod(dptr, host)
        for mode in ("device", "host"):
            best = None
            for rep in range(3):
                sim.reset(); sim.flush_l2(); sim.synchronize()
                t0 = time.perf_counter()
                for k in range(nb):
                    if mode == "device":
                        sim.upload_batch_las_device(dptr + k * BATCH * bpp, BATCH, layout)
                    else:
                        sim._check(sim._lib.simlod_upload_batch_las(sim._ctx, hptr + k * BATCH * bpp, BATCH, ctypes.byref(layout)))
                sim.synchronize()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            key = "value" if mode == "device" else "e2e"
            out[key] = {"value": round(n / best / 1e6, 1), "unit": "Mpoints/s",
                        "how": "records resident in HBM" if mode == "device" else "records in pinned host memory, H2D inside the timed region"}
        got = sim.ring_slot(nb - 1, 1000)
        want = oracle.decode_las(recs[nb - 1][:1000], 1000, bpp, 2, scale, offset)
        assert (got == want).all()
        out["roofline"] = {"bound": "hbm", "algorithmic_bytes_per_point": bpp + 16,
                           "achieved_gbs": round(out["value"]["value"] * 1e6 * (bpp + 16) / 1e9, 1)}
    finally:
        sim.close()
    if oracle.ref_las() is not None:
        d = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
        path = os.path.join(d, "simlod_bench_%d.las" % os.getpid())
        try:
            data.write_las(path, np.concatenate(host_batches), 2, scale, offset)
            best = None
            for threads in sorted({1, min(8, os.cpu_count() or 1), os.cpu_count() or 1}):
                dt_t = oracle.ref_las_bench(path, n, 250_000, threads)
                if best is None or dt_t < best[0]:
                    best = (dt_t, threads)
            dt, threads = best
            out["cpu_baseline"] = {"value": round(n / dt / 1e6, 1), "unit": "Mpoints/s", "cores": threads, "kind": "reference",
                                   "sample": "loadLasNative (LasLoader.cpp compiled from /root/reference) on %d M points from tmpfs in 250k-point batches, long-lived loader threads; best of 1 / 8 / all cores" % (n // 1000000)}
        finally:
            if os.path.exists(path):
                os.remove(path)
    return out


def bench_stream_file(sim_device, host_batches, mn, mx):
    """.simlod file (tmpfs, and cold from disk when the box has one) -> loader threads -> pinned pool -> ring -> octree, with
    the reference's own loadFileNative (SimlodLoader.cpp compiled from /root/reference) timed beside it on the host cores."""
    import tempfile
    import oracle
    from simlod_b200 import SimLOD, data
    nb = len(host_batches)
    n = nb * BATCH
    d = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    path = os.path.join(d, "simlod_bench_%d.simlod" % os.getpid())
    out = {"points": n, "file_bytes": 24 + 16 * n}
    try:
        data.write_simlod(path, np.concatenate(host_batches), mn, mx)
        sim = SimLOD(320, 176, device=sim_device, persistent_bytes=max(4 << 30, nb * (220 << 20)))
        try:
            best = None
            threads = min(16, os.cpu_count() or 8)
            for rep in range(3):
                t0 = time.perf_counter()
                got, kms, tms = sim.insert_simlod_file(path, loader_threads=threads)
                dt = time.perf_counter() - t0
                assert got == n and sim.stats().numPoints == n
                if best is None or dt < best[0]:
                    best = (dt, kms, tms)
            out["e2e"] = {"value": round(n / best[0] / 1e6, 1), "unit": "Mpoints/s", "how": "wall clock incl. reset, %d loader threads, file in tmpfs" % threads,
                          "device_ms": round(best[2], 3), "kernel_ms": round(best[1], 3)}
        finally:
            sim.close()
        if oracle.ref_simlod() is not None:
            best = None
            for threads in sorted({1, min(8, os.cpu_count() or 1), os.cpu_count() or 1}):
                dt_t = oracle.ref_simlod_bench(path, n, BATCH, threads)
                if best is None or dt_t < best[0]:
                    best = (dt_t, threads)
            out["cpu_baseline"] = {"value": round(n / best[0] / 1e6, 1), "unit": "Mpoints/s", "cores": best[1], "kind": "reference",
                                   "sample": "loadFileNative (SimlodLoader.cpp compiled from /root/reference), %d x 1M-point reads from tmpfs into host memory; best of 1 / 8 / all cores" % nb}
        # cold file: the same scan on a disk-backed file system, its pages evicted before every run, read unbuffered (O_DIRECT)
        cold_path = os.path.join(tempfile.gettempdir(), "simlod_bench_cold_%d.simlod" % os.getpid())
        try:
            data.write_simlod(cold_path, np.concatenate(host_batches), mn, mx)

            def evict():
                fd = os.open(cold_path, os.O_RDONLY)
                try:
                    os.fsync(fd); os.posix_fadvise(fd, 0, 0, os.POSIX_FADV_DONTNEED)
                finally:
                    os.close(fd)
            sim = SimLOD(320, 176, device=sim_device, persistent_bytes=max(4 << 30, nb * (220 << 20)))
            try:
                cold = {}
                for mode, direct in (("direct", True), ("buffered", False)):
                    best = None
                    try:
                        for rep in range(2):
                            evict()
                            t0 = time.perf_counter()
                            got, kms, tms = sim.insert_simlod_file(cold_path, loader_threads=min(16, os.cpu_count() or 8), direct=direct)
                            dt = time.perf_counter() - t0
                            assert got == n and sim.stats().numPoints == n
                            best = dt if best is None else min(best, dt)
                        cold[mode] = round(n / best / 1e6, 1)
                    except Exception as e:
                        cold[mode] = repr(e)[:160]
                cold["how"] = "file on %s, page cache evicted (fsync + POSIX_FADV_DONTNEED) before every run; Mpoints/s wall clock incl. reset" % tempfile.gettempdir()
                out["cold_file"] = cold
            finally:
                sim.close()
        finally:
            if os.path.exists(cold_path):
                os.remove(cold_path)
    finally:
        if os.path.exists(path):
            os.remove(path)
    return out


def dump_outputs(sim, out_dir):
    """What a caller of the timed path receives, reduced to what is the same from run to run (DESIGN.md §3): the
    deterministic Stats fields and the octree's canonical form (per node, in (level, X, Y, Z) order: counters, chunk
    counts, and the hashes of its sorted points and voxel positions as 32-bit halves), all exact in float64."""
    import oracle
    os.makedirs(out_dir, exist_ok=True)
    st = sim.stats()
    rec = oracle.canon_from_image(*sim.download_octree()).records
    cols = ("level", "X", "Y", "Z", "counter", "numPoints", "numVoxels", "numVoxelsStored", "isLeaf", "chunksPoints", "chunksVoxels")
    halves = [(rec[f] >> np.uint64(s)) & np.uint64(0xFFFFFFFF) for f in ("hashPoints", "hashVoxelPos") for s in (32, 0)]
    np.save(os.path.join(out_dir, "stats.npy"), np.array([int(getattr(st, f)) for f in oracle.STATS_FIELDS], dtype=np.float64))
    np.save(os.path.join(out_dir, "octree_nodes.npy"), np.stack([rec[c].astype(np.float64) for c in cols], axis=1))
    np.save(os.path.join(out_dir, "octree_hashes.npy"), np.stack([h.astype(np.float64) for h in halves], axis=1))


def run_reference(args, rank, world):
    """The reference's algorithm on the host cores: oracle port (the reference has no CPU octree builder to compile; its
    kernels need a GPU). Same workload (the 350 M-point stream of the numpy generator the device generator restates
    bit for bit); one step = one full 1 M-point batch, a bounded sample of K steps from reset."""
    if rank != 0:
        return
    import oracle
    from simlod_b200 import data
    W, K = max(args.warmup, 0), max(args.steps, 1)
    nb = args.batches
    n_total = nb * BATCH
    K = min(K, nb)
    batches = [data.terrain(n_total, b * BATCH, BATCH, seed=TERRAIN_SEED)[0] for b in range(max(K, min(W, nb)))]
    mn, mx = (0.0, 0.0, 0.0), data.TERRAIN_EXTENT
    o = oracle.Oracle(mn, mx)
    for b in batches[:W]:
        o.add_batch(b)
    o = oracle.Oracle(mn, mx)
    t0 = time.perf_counter()
    for b in batches[:K]:
        o.add_batch(b)
    dt = time.perf_counter() - t0
    s = o.stats()
    assert s.numPoints == K * BATCH
    val = K * BATCH / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mpoints/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32+f32",
        "data": "synthetic",
        "config": {"workload": workload_name(nb),
                   "note": "reference algorithm restated for the CPU (oracle/oracle.cpp); the reference itself has no CPU builder. Bounded sample: the first %d batches of the stream from reset" % K},
        "cpu_baseline": {"value": val, "unit": "Mpoints/s", "cores": 1, "kind": "port", "sample": "the first %d of the %d batches of rank 0's stream, from reset" % (K, nb)},
        "e2e": {"value": val, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def bench_merged_octree(sim, dptr, nb_avail, rank, world, dev, barrier):
    """SURVEY.md §8f-3 beside the batch-sharded headline: ONE octree over the N GPUs. Every rank sends the points of its
    first 16 batches to the owners of their level-2 cells (fused partition + push kernel over NVLink peer memory,
    DESIGN.md §9.3), the exchange of group g+1 enqueued before the insertion of group g, and inserts what it receives.
    Every local step is followed by an agreement (all ranks ok?) before the next collective, so a rank that cannot run it
    makes all ranks skip the leg instead of hanging the others."""
    import torch
    import torch.distributed as dist
    from simlod_b200 import dist as sdist
    K, LEVEL, DEPTH = min(16, nb_avail), 2, 8

    def agree(ok):
        t = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(int(t.item()))

    err = None
    try:
        plan0 = sim.partition_plan(LEVEL, np.zeros(8 ** LEVEL, np.uint8), world)
        hist = np.zeros(8 ** LEVEL, np.int64)
        for i in range(K):
            hist += sim.partition_count(dptr + i * BATCH * 16, BATCH, plan0)[1].astype(np.int64)
    except Exception as e:
        err = repr(e)
    if not agree(err is None):
        return {"error": err or "another rank failed while planning"}
    t = torch.tensor(hist, device=dev)
    dist.all_reduce(t)
    owners = sdist.plan_owners(t.cpu().numpy(), world)
    ex = None
    try:
        ex = sdist.SpatialExchange(sim, LEVEL, owners, capacity_points=BATCH, depth=DEPTH, mode="p2p", device=torch.device(dev), timeout_ms=5000)
    except Exception as e:
        err = repr(e)
    if not agree(err is None):
        return {"error": err or "another rank could not set up peer memory"}
    groups = [[(dptr + i * BATCH * 16, BATCH) for i in range(g0, min(K, g0 + DEPTH))] for g0 in range(0, K, DEPTH)]
    best, received = None, 0
    for rep in range(3):
        try:
            sim.reset()
            barrier()
            t0 = time.perf_counter()
            ex.prepare([bt for g in groups for bt in g])
            ex.send_group(groups[0])
            received = 0
            for gi in range(len(groups)):
                ptr, n = ex.wait_group()
                if gi + 1 < len(groups):
                    ex.send_group(groups[gi + 1])
                if n:
                    sim.insert_device(ptr, n)
                received += n
            sim.synchronize()
        except Exception as e:
            err = repr(e)
        if not agree(err is None):
            return {"error": err or "another rank failed during the exchange"}
        barrier()
        dt = sdist.max_over_ranks(time.perf_counter() - t0, dev)
        best = dt if best is None else min(best, dt)
    st = sim.stats()
    tot = sdist.reduce_stats(st, dev)
    return {"value": round(world * K * BATCH / best / 1e6, 2), "unit": "Mpoints/s",
            "what": "ONE octree over %d GPUs: %d x 1M-point batches per GPU exchanged by owner of the level-%d cell (fused partition + push over NVLink peer memory, groups of %d batches, "
                    "exchange of group g+1 under the insertion of group g) and inserted; host clock around barriers, best of 3, planning window included" % (world, K, LEVEL, DEPTH),
            "points_total": world * K * BATCH, "numPoints_all_ranks": tot["numPoints"], "all_points_arrived": tot["numPoints"] == world * K * BATCH,
            "received_this_rank": int(received), "bit_exactness": "tests/test_merged_octree.py, tools/bench_merged.py (every rank's octree vs a local rebuild)"}


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE line, the JSON result: whatever libraries print on fd 1 meanwhile (NCCL's version banner, a
    device-side printf of the reference's reset kernel) goes to stderr."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from simlod_b200 import SimLOD, data
    from simlod_b200 import dist as sdist

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = "cuda:%d" % local_rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    NB = args.batches
    W, K = max(args.warmup, 0), min(max(args.steps, 1), NB)
    passes = max(args.passes, 1)
    npts = K * BATCH                                         # timed points per pass: the first K batches of the stream
    nb_gen = max(K, min(W, NB), min(16, NB))                 # batches generated: timed, warm-up and the CPU legs' sample
    mn, mx = (0.0, 0.0, 0.0), data.TERRAIN_EXTENT
    peak, peak_src = peaks()

    import oracle          # the reference kernels' scratch needs 408.8 MB of momentary buffer; ours fits 300 MB either way
    sim = SimLOD(W_PX, H_PX, device=local_rank, persistent_bytes=max(8 << 30, K * (72 << 20)))
    sampler = ClockSampler(local_rank)
    sampler.start()
    windows = []
    try:
        sim.set_box(mn, mx)
        # this rank's stream (tile `rank` of the survey), generated on the device; a pinned host copy for the e2e leg
        t_gen = time.time()
        dptr = sim.device_alloc(nb_gen * BATCH * 16)
        sim.generate(sim.GEN_TERRAIN, dptr, NB * BATCH, 0, nb_gen * BATCH, TERRAIN_SEED + rank)
        host_ptr = sim.host_alloc(npts * 16)
        numa_node = sim.numa_node()
        sim._check(sim._lib.simlod_memcpy_dtoh(sim._ctx, host_ptr, dptr, npts * 16))
        t_gen = time.time() - t_gen

        # warm-up: W batches (code, clocks, allocator paths), then start over
        sim.reset()
        if W:
            sim.insert_device(dptr, min(W, NB) * BATCH)
        info0 = sim.launch_info()

        # ---- timed region 1: inputs resident in HBM, median of `passes` passes over the whole stream ----------
        ks, ts = timed_passes(sim, lambda: sim.insert_device(dptr, npts), npts, passes, barrier, windows)
        st = sim.stats()
        info1 = sim.launch_info()
        launches_per_pass = (info1["launches"] - info0["launches"]) // passes - 2     # minus the reset kernel and the L2 flush fill
        b = sim.buffers()
        ctl = sim.memcpy_dtoh(b.momentary + 80, 16).view(np.uint64)    # Ctl::spilledTotal, voxelsTotal (construct.cu)
        spilled_total, voxels_total = int(ctl[0]), int(ctl[1])
        kernel_ms = float(np.median(ks))
        t_value = sdist.max_over_ranks(float(np.median(ts)), dev)
        t_kernel = sdist.max_over_ranks(kernel_ms, dev)
        totals = sdist.reduce_stats(st, dev)
        if args.dump_outputs and rank == 0:
            dump_outputs(sim, args.dump_outputs)

        # ---- render on the built octree (rank-local; reported at rank 0) --------------------------
        render = None
        if not args.no_render and rank == 0:
            t0 = time.time()
            render = render_sweep(sim, mx, peak)
            render["metric"] = "render Msamples/s @1GPU (1920x1080), 6 cameras on the %d M-point octree" % K
            render["render_blocks"] = sim.launch_info()["render_blocks"]
            windows.append((t0, time.time()))

        # ---- the reference's own kernels on this GPU (rank 0, N = 1) ---------------------------------
        reference_gpu = None
        if rank == 0 and world == 1 and not args.no_reference_gpu:
            t0 = time.time()
            reference_gpu = bench_reference_gpu(local_rank, dptr, K, (mn, mx), peak, sim)
            windows.append((t0, time.time()))
            reference_gpu["clocks"] = sampler.summary([windows[-1]])

        # ---- timed region 2: end to end from pinned host memory (median of 3 passes) ----------------------
        info2 = sim.launch_info()
        e_passes = min(3, passes)
        eks, ets = [], []
        e_wall = []
        for _ in range(e_passes):
            sim.reset()
            sim.flush_l2()
            barrier()
            t0 = time.time()
            e_kernel_ms, e_total_ms = sim.insert_host_ptr(host_ptr, npts)
            st_e = sim.stats()                                  # device->host read of the result
            barrier()
            t1 = time.time()
            windows.append((t0, t1))
            assert st_e.numPointsProcessed == npts and st_e.numPoints == npts
            eks.append(e_kernel_ms); ets.append(e_total_ms); e_wall.append((t1 - t0) * 1e3)
        info3 = sim.launch_info()
        e_launches = (info3["launches"] - info2["launches"]) // e_passes - 2
        t_e2e = sdist.max_over_ranks(float(np.median(ets)), dev)
        t_e2e_wall = sdist.max_over_ranks(float(np.median(e_wall)), dev)

        # a bounded host sample of the same stream for the CPU legs (rank 0, N = 1)
        sample_batches = []
        if rank == 0 and world == 1:
            nb_s = min(16, nb_gen)
            raw = sim.memcpy_dtoh(dptr, nb_s * BATCH * 16).view(data.POINT_DTYPE)
            sample_batches = [raw[i * BATCH:(i + 1) * BATCH] for i in range(nb_s)]
        # ---- one octree over the N GPUs (SURVEY.md §8f-3), N > 1 only ----------------------------------------
        merged = None
        if world > 1 and not args.no_extras:
            t0 = time.time()
            try:
                sim.set_box(mn, mx)
                merged = bench_merged_octree(sim, dptr, nb_gen, rank, world, dev, barrier)
            except Exception as e:
                merged = {"error": repr(e)}
            windows.append((t0, time.time()))
        sim.device_free(dptr)
        sim.host_free(host_ptr)

        # ---- BASELINE.json configs[3] as specified: one N x 250 M shell, round-robin batches ----------------
        config4 = None
        if not args.no_extras:
            try:
                nb4 = min(CONFIG4_BATCHES_PER_GPU, NB)          # (the developer knob --batches shrinks this leg too)
                total4 = world * nb4
                d4 = sim.device_alloc(nb4 * BATCH * 16)
                for k, bidx in enumerate(sdist.shard_batches(total4, rank, world)):
                    sim.generate(sim.GEN_SHELL, d4 + k * BATCH * 16, total4 * BATCH, bidx * BATCH, BATCH, SHELL_SEED)
                sim.set_box((0.0, 0.0, 0.0), (data.SHELL_CUBE,) * 3)
                ks4, ts4 = timed_passes(sim, lambda: sim.insert_device(d4, nb4 * BATCH), nb4 * BATCH, min(3, passes), barrier, windows)
                st4 = sim.stats()
                t4 = sdist.max_over_ranks(float(np.median(ts4)), dev)
                tk4 = sdist.max_over_ranks(float(np.median(ks4)), dev)
                tot4 = sdist.reduce_stats(st4, dev)
                config4 = {"workload": "sphere shell R=1800 in a 4096^3 cube, %d M points in lat/lon tile order, rank g inserts the 1M-point batches b = g (mod %d): %d M points per GPU" % (total4, world, nb4),
                           "value": round(world * nb4 * BATCH / t4 / 1e3, 2), "unit": "Mpoints/s", "kernel_only": round(world * nb4 * BATCH / tk4 / 1e3, 2),
                           "passes": min(3, passes), "octree": {k: tot4[k] for k in ("numNodes", "numPoints", "numVoxels")},
                           "note": "per-GPU work changes with N here: a G-times sparser sample of a G-times denser shell has more nodes and voxels per point (DESIGN.md §8); `value` above keeps per-GPU work fixed instead"}
                sim.device_free(d4)
                sim.set_box(mn, mx)
            except Exception as e:          # reported, never fatal for the headline
                config4 = {"error": repr(e)}
    finally:
        sampler.stop()
    sim.close()

    # ---- "next" rows (SURVEY.md §8f-1/2), rank 0 at N = 1 -------------------------------------------------
    las = stream = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            las = bench_las(local_rank, sample_batches[:8], mn, mx)
        except Exception as e:
            las = {"error": repr(e)}
        try:
            stream = bench_stream_file(local_rank, sample_batches, mn, mx)
        except Exception as e:
            stream = {"error": repr(e)}

    # ---- CPU baseline (rank 0, N = 1 only): oracle port on a bounded sample -----------------------
    cpu = None
    if rank == 0 and world == 1:
        nb_c = min(args.cpu_sample_batches, len(sample_batches))
        o = oracle.Oracle(mn, mx)
        t0 = time.perf_counter()
        for bt in sample_batches[:nb_c]:
            o.add_batch(bt)
        dt = time.perf_counter() - t0
        cpu = {"value": round(nb_c * BATCH / dt / 1e6, 4), "unit": "Mpoints/s", "cores": 1, "kind": "port",
               "sample": "first %d of the %d batches of the same stream, oracle/oracle.cpp, %.1f s" % (nb_c, NB, dt)}

    if rank == 0:
        all_pts = world * npts
        value = all_pts / t_value / 1e3
        s_frac = spilled_total / npts
        v_frac = voxels_total / npts
        alg_bytes = (32.0 + 32.0 * s_frac + 16.0 * v_frac) * npts          # this rank, one pass
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = recorded_traffic(K)
        n_launch = max(launches_per_pass, 1)
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "Mpoints/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(t_value / K, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32+f32", "data": "synthetic",
            "config": {"workload": workload_name(NB),
                       "batch_points": BATCH, "points_per_gpu": npts, "steps_per_pass": K, "timed_passes": passes,
                       "timing": "median of %d passes, each the first %d batches of the %d-batch stream from reset (a step = one 1M-point batch); max over ranks of the per-rank median" % (passes, K, NB),
                       "parallelism": "batch-sharded x%d (one %d-batch scan tile per GPU, no data-path collective)" % (world, NB),
                       "l2": "inputs %d MB > L2 (126 MB); L2 flushed before each timed pass" % (npts * 16 // 1000000),
                       "kernel_only_mpoints_per_s": round(all_pts / t_kernel / 1e3, 2),
                       "pass_ms": [round(x, 3) for x in ts], "pass_kernel_ms": [round(x, 3) for x in ks],
                       "octree": {k: totals[k] for k in ("numNodes", "numInner", "numLeaves", "numPoints", "numVoxels", "allocatedBytes_persistent")},
                       "construct_blocks": info1["construct_blocks"], "datagen_s": round(t_gen, 1),
                       "data_generator": "simlod_generate (csrc/gen.cu), bit-identical to simlod_b200/data.py:terrain (tests/test_generators.py)"},
            "roofline": {"bound": "hbm", "kernel": "kernel_construct", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 5),
                         "traffic": traffic.get("dram_bytes_per_launch") if traffic else None,
                         "traffic_source": traffic.get("source") if traffic else None,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_point": round(alg_bytes / npts, 3), "spilled_fraction_s": round(s_frac, 4),
                         "voxels_per_point_v": round(v_frac, 4), "launches": launches_per_pass,
                         "avg_launch_ms": round(kernel_ms / n_launch, 4), "algorithmic_bytes_per_launch": round(alg_bytes / n_launch),
                         "note": "latency/atomic bound, not bandwidth bound: see DESIGN.md §7"},
            "e2e": {"value": round(all_pts / t_e2e / 1e3, 2), "unit": "Mpoints/s", "h2d_bytes_per_step": BATCH * 16,
                    "d2h_bytes_per_step": round(112.0 * (e_launches + 1) / K, 1), "wall_clock_value": round(all_pts / t_e2e_wall / 1e3, 2),
                    "launches": e_launches, "passes": e_passes, "pinned_on_numa_node": numa_node},
            "gpu_launches": launches_per_pass * passes,
            "clocks": sampler.summary(windows),
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if reference_gpu:
            line["reference_gpu"] = reference_gpu
        if render:
            line["render"] = render
        if config4:
            line["config4"] = config4
        if merged:
            line["merged_octree"] = merged
        if las:
            line["las_decode"] = las
        if stream:
            line["stream_file"] = stream
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
