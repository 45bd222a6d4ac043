#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 descriptor matcher; prints one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one whole matcher call over one synthetic descriptor pair of the named BASELINE.json
configuration: descriptor upload/packing + forward kNN (+ reverse kNN for mutual) + filter.
  value : queries/s, descriptors (AoS, as PCL lays them out) already resident in HBM; CUDA events.
  e2e   : the same through the host-facing C-ABI (b200m_upload from pinned host memory, result
          records copied back to the host) -- host<->device copies inside the timed region.
Multi-GPU (torchrun, one rank per GPU): source rows (and, for the mutual pass, target rows) are sharded
across ranks, both descriptor sets replicated; one NCCL all-gather of the reverse table; strong scaling.
`--impl reference` times the reference's CPU matcher semantics (the oracle port; the reference itself
cannot be built here: PCL/OpenCV/FLANN absent) on the host cores, bounded sample per step.
`--dump-outputs DIR` writes what the last timed step returned (see write_outputs); the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (descriptor, n_src, n_tgt, k, mode, BASELINE.json config string)
    "c1": ("fpfh", 20000, 20000, 1, "mutual", "FPFH-33 20k x 20k k=1 mutual (BASELINE configs[0])"),
    "c2": ("fpfh", 200000, 200000, 2, "ratio", "FPFH-33 200k x 200k k=2 + ratio 1.1 (BASELINE configs[1])"),
    "c3": ("shot", 500000, 500000, 2, "mutual", "SHOT-352 500k x 500k k=2 + mutual (BASELINE configs[2])"),
    "c3s": ("shot", 40000, 40000, 2, "mutual", "SHOT-352 40k x 40k k=2 + mutual (reduced copy of configs[2], for debugging)"),
    "c4": ("fpfh", 2000000, 2000000, 5, "mutual", "FPFH-33 2M x 2M k=5 mutual k-lists (BASELINE configs[3])"),
    # configs[4]: the target set is sharded 1M rows per GPU (8M at 8 GPUs) and every rank holds all queries; per-rank exact
    # top-k with global indices, one NCCL all-gather of the k-lists, merge kernel.  n_tgt here is PER RANK (weak scaling).
    "c5": ("shot", 500000, 1000000, 2, "knn_target_sharded",
           "SHOT-352 kNN k=2, 500k queries x (1M target rows per GPU), target-sharded + NCCL top-k merge (BASELINE configs[4])"),
}
METRICS = {
    "c1": "descriptor queries/sec (FPFH-33 k=1 + mutual)",
    "c2": "descriptor queries/sec (FPFH-33 k=2 + ratio)",
    "c3": "descriptor queries/sec (k=2 + mutual)",          # BASELINE.json's metric string, quoted on configs[2]
    "c3s": "descriptor queries/sec (k=2 + mutual, reduced size)",
    "c4": "descriptor queries/sec (FPFH-33 k=5 + mutual)",
    "c5": "descriptor queries/sec (SHOT-352 k=2 kNN, target-sharded)",
}


def ncu_traffic(wl):
    """dram__bytes_read.sum + dram__bytes_write.sum per candidate-kernel launch, read at run time from the committed ncu
    --set full summary of the same workload on 1 GPU (profiles/ncu_traffic.json names the summary file per workload;
    tools/ncu_traffic.py regenerates it from the .ncu-rep).  None when there is no capture."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        e = json.load(open(p)).get(wl)
    except Exception:
        return None, None
    if not e:
        return None, None
    return float(e["bytes_per_launch"]), "%s (%s)" % (e["source"], e.get("note", "ncu --set full, 1 GPU"))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_sustained": d.get("bf16_tflops_sustained", 1388.3), "bf16_burst": d.get("bf16_tflops", 1658.5),
                "hbm": d.get("hbm_gbs", 6450.3), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "B200_PROFILING.md fallback (of fallback)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region.  The sampler process is started before the
    warm-up (nvidia-smi needs a few hundred ms before its first line) and streams a time-stamped line every 20 ms;
    stop() keeps the lines whose time stamps fall inside the timed region's host-clock window."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.t_begin = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def begin(self):
        """Call right before the timed region starts (after the barrier)."""
        self.t_begin = time.time()

    @staticmethod
    def _stamp(text):
        import datetime
        return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()

    def stop(self):
        t_end = time.time()
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(",") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        parsed = []
        for r in rows:
            try:
                try:
                    ts = self._stamp(r[0])
                except Exception:
                    ts = t_end   # unparsable time stamp: count the line as inside the window
                parsed.append((ts, float(r[1]), float(r[2]), float(r[3]),
                               [n for n, v in zip(names, r[4:8]) if v.strip().lower() == "active"]))
            except Exception:
                pass
        if not parsed:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        t0 = self.t_begin if self.t_begin is not None else parsed[0][0]
        window = "timed region"
        inside = [q for q in parsed if t0 <= q[0] <= t_end]
        if not inside:
            # a timed region shorter than the sampling period: the samples closest to it (the warm-up runs the same
            # steps back to back, so these are still samples under load)
            mid = 0.5 * (t0 + t_end)
            inside = sorted(parsed, key=lambda q: abs(q[0] - mid))[:3]
            window = "nearest samples (timed region of %.0f ms is shorter than the sampling period)" % (1e3 * (t_end - t0))
        reasons = set()
        for q in inside:
            reasons.update(q[4])
        return {"sm_mhz": float(np.median([q[1] for q in inside])), "sm_max_mhz": float(max(q[2] for q in inside)),
                "power_w_max": float(max(q[3] for q in inside)), "samples": len(inside), "window": window,
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
class CpuReference:
    """Oracle (CPU port of the reference matcher) on a bounded query sample against the FULL opposite
    set, both directions for mutual.  Data are generated once per process."""

    def __init__(self, desc, n_src, n_tgt, k, mode):
        from lidar_global_registration_b200 import synth
        from oracle import oracle as orc
        self.orc, self.k, self.both = orc, k, mode == "mutual"
        try:
            orc.set_num_threads(len(os.sched_getaffinity(0)))   # all host cores, whatever OMP_NUM_THREADS torchrun exported
        except AttributeError:
            orc.set_num_threads(os.cpu_count() or 1)
        self.cores = orc.num_threads()
        self.n_src, self.n_tgt = n_src, n_tgt
        # numpy generation is slow at the named sizes: generate <= 200k rows and tile them with small
        # perturbations up to the named row counts (the CPU cost per query only depends on the row counts)
        n_gen_s, n_gen_t = min(n_src, 200000), min(n_tgt, 200000)
        src, tgt, dim = synth.make_pair(desc, n_gen_s, n_gen_t, nan_frac=0.001)
        rng = np.random.default_rng(11)

        def tile(a, n):
            a = np.ascontiguousarray(a[:, :dim])
            if a.shape[0] >= n:
                return a[:n]
            reps = (n + a.shape[0] - 1) // a.shape[0]
            return np.concatenate([a * np.float32(1 + 1e-3 * rng.standard_normal()) for _ in range(reps)])[:n]
        self.s, self.t, self.dim = tile(src, n_src), tile(tgt, n_tgt), dim
        self.probe = max(self.cores * 4, 64)
        self.t_probe = self._run(self.probe)

    def _run(self, nq):
        t0 = time.perf_counter()
        self.orc.knn(self.s[:nq], self.t, self.k)
        if self.both:
            self.orc.knn(self.t[:nq], self.s, self.k)
        return time.perf_counter() - t0

    def rate(self, budget_s):
        nq = int(max(self.probe, min(self.n_src, self.probe * budget_s / max(self.t_probe, 1e-6))))
        secs = self._run(nq)
        for _ in range(2):   # the probe includes thread start-up: re-aim once or twice if the sample came out short
            if secs >= 0.4 * budget_s or nq >= self.n_src:
                break
            nq = int(min(self.n_src, nq * 0.8 * budget_s / max(secs, 1e-6)))
            secs = self._run(nq)
        sample = "%d source queries vs all %d target rows%s (D=%d, k=%d), oracle port of the reference matcher, OpenMP" % (
            nq, self.n_tgt, (" + %d target queries vs all %d source rows" % (nq, self.n_src)) if self.both else "",
            self.dim, self.k)
        return nq / secs, self.cores, sample, secs


def opencv_knn(q, t, k, block=10000):
    """k nearest train rows of every query row with cv2.BFMatcher(NORM_L2).knnMatch over train blocks of `block` rows, the
    per-block lists merged in block order (stable: an earlier block's entry stays in front of an equal later one) ->
    (idx [nq, k] int64, -1 padded; dist [nq, k] float32, +inf padded).  tests/test_bench_host.py checks it against the oracle."""
    import cv2
    matcher = cv2.BFMatcher(cv2.NORM_L2)
    nq = q.shape[0]
    bd = np.full((nq, k), np.inf, np.float32)
    bi = np.full((nq, k), -1, np.int64)
    for t0 in range(0, t.shape[0], block):
        res = matcher.knnMatch(q, t[t0:t0 + block], k)
        d = np.full((nq, k), np.inf, np.float32)
        i = np.full((nq, k), -1, np.int64)
        for r, lst in enumerate(res):
            for c, m in enumerate(lst):
                d[r, c], i[r, c] = m.distance, m.trainIdx + t0
        alld, alli = np.concatenate([bd, d], 1), np.concatenate([bi, i], 1)
        order = np.argsort(alld, 1, kind="stable")[:, :k]
        bd, bi = np.take_along_axis(alld, order, 1), np.take_along_axis(alli, order, 1)
    return bi, bd


def opencv_bfmatcher_rate(ref, budget_s, block=10000):
    """The third-party routine the reference's matchBF calls -- cv::BFMatcher(NORM_L2).knnMatch, here through Python's cv2 -- in
    the reference's blocking (bf_block_size = 10000 train rows per call, include/matching.h:594-634) with the per-block results
    merged into k-lists, on a bounded query sample against the full opposite set (both directions for mutual).  Not the
    reference (PCL / OpenCV C++ cannot be built in this image), but its actual arithmetic kernel with OpenCV's own SIMD and
    threads; None where cv2 is not installed."""
    try:
        import cv2
    except ImportError:
        return None
    cv2.setNumThreads(ref.cores)

    def run(nq):
        t_0 = time.perf_counter()
        opencv_knn(ref.s[:nq], ref.t, ref.k, block)
        if ref.both:
            opencv_knn(ref.t[:nq], ref.s, ref.k, block)
        return time.perf_counter() - t_0
    nq = max(ref.cores * 8, 128)
    secs = run(nq)
    nq = int(max(nq, min(ref.n_src, block, nq * 0.8 * budget_s / max(secs, 1e-6))))
    secs = run(nq)
    return {"value": nq / secs, "unit": "queries/s", "threads": cv2.getNumThreads(), "opencv": cv2.__version__, "seconds": secs,
            "sample": "%d source queries vs all %d target rows%s, cv2.BFMatcher(NORM_L2).knnMatch in train blocks of %d rows + merge"
                      % (nq, ref.n_tgt, (" + %d target queries vs all %d source rows" % (nq, ref.n_src)) if ref.both else "", block)}


def run_reference(args, wl):
    desc, n_src, n_tgt, k, mode, cfg = WORKLOADS[wl]
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = CpuReference(desc, n_src, n_tgt, k, mode)
    rates, secs_all = [], []
    sample, cores = "", ref.cores
    for i in range(args.warmup + args.steps):
        r, cores, sample, secs = ref.rate(6.0)
        if i >= args.warmup:
            rates.append(r)
            secs_all.append(secs)
    value = float(np.mean(rates))
    engine = "oracle port of the reference matcher (C, OpenMP)"
    ocv = opencv_bfmatcher_rate(ref, 6.0)
    port_value = value
    if ocv and ocv["value"] > value:   # the line carries the FASTER of the two CPU engines
        value, sample, engine = ocv["value"], ocv["sample"], "cv2.BFMatcher (the routine the reference's matchBF calls), reference blocking"
        secs_all = [ocv["seconds"]]
    line = {"impl": "reference", "metric": METRICS[wl], "value": value, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(secs_all)),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(wl, max(args.gpus, 1)),
            "timing": "wall clock around the CPU matcher call, bounded query sample per step",
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample, "engine": engine,
                             "oracle_port_value": port_value, "opencv_bfmatcher": ocv},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


DIMS = {"fpfh": (33, 132), "shot": (352, 1444), "rops": (135, 540)}   # descriptor length, sizeof(FeatureT) as PCL lays it out


def measure_local(torch, D, M, synth, dev, timed, n=200000, k=2, radius=2.5, box=100.0):
    """queries/s of the guess-gated kNN (b200m_knn_local_device), descriptors and keypoints resident in HBM: FPFH-33
    n x n, keypoints uniform in a box^3 cube (about n * 4/3 pi r^3 / box^3 = 13 train keypoints pass each query's gate)."""
    import ctypes as C
    src, tgt, dim = synth.make_pair_torch("fpfh", n, n, dev)
    g = torch.Generator(device=dev)
    g.manual_seed(566)
    qx = torch.zeros((n, 4), device=dev)
    tx = torch.zeros((n, 4), device=dev)
    qx[:, :3] = torch.rand((n, 3), device=dev, generator=g) * box
    tx[:, :3] = torch.rand((n, 3), device=dev, generator=g) * box
    idx = torch.empty((n, k), dtype=torch.int32, device=dev)
    dst = torch.empty((n, k), dtype=torch.float32, device=dev)
    cnt = torch.empty((n,), dtype=torch.int32, device=dev)
    out = {"metric": "descriptor queries/sec (FPFH-33 k=2, matchLocal with match_search_radius)", "unit": "queries/s",
           "config": {"workload": "FPFH-33 %d x %d k=%d, 3-D gate radius %.1f in a %.0f^3 cube (matchLocal, include/matching.h:637-678)"
                                  % (n, n, k, radius, box), "n_src": n, "n_tgt": n, "k": k}}
    for label, min_rows in (("cell_list", "1"), ("gate_against_all_rows", "1000000000")):
        os.environ["B200M_LOCAL_MIN_ROWS"] = min_rows
        be = D.GpuBackend(dev.index)
        try:
            be.upload_device(0, src, dim)
            be.upload_device(1, tgt, dim)
            p = be.ctx._params(k, M.MODE_KNN_ONLY)
            v = C.c_void_p

            def step():
                be.ctx._ck(be.ctx._L.b200m_knn_local_device(be.ctx._h, C.byref(p), 0, v(qx.data_ptr()), v(tx.data_ptr()), 16,
                                                            float(radius), v(idx.data_ptr()), v(dst.data_ptr()), v(cnt.data_ptr())))
                return None, cnt
            for _ in range(2):
                step()
            steps = 5 if label == "cell_list" else 2
            ms, o = timed(step, steps)
            out[label] = {"value": n * steps / (ms * 1e-3), "ms_per_call": ms / steps, "neighbours_found_per_query": float(cnt.float().mean().item())}
        finally:
            be.close()
    os.environ.pop("B200M_LOCAL_MIN_ROWS", None)
    out["value"] = out["cell_list"]["value"]
    return out


def workload_config(wl, world):
    """`config` of a workload: identical on both arms (the driver compares them), nothing run-specific in it."""
    desc, n_src, n_tgt, k, mode_name, cfg = WORKLOADS[wl]
    dim, stride_b = DIMS[desc]
    tsharded = mode_name == "knn_target_sharded"
    return {"workload": cfg, "descriptor": desc, "dim": dim, "n_src": n_src, "n_tgt": n_tgt, "k": k, "filter": mode_name,
            "row_stride_bytes": stride_b,
            "sharding": (("target-sharded (n_tgt rows per rank, %d in total), queries replicated, NCCL all-gather + merge"
                          % (n_tgt * world)) if tsharded else
                         ("query-sharded, target replicated" if world > 1 else "single GPU")),
            "l2": ("inputs larger than L2 (no flush needed)" if n_tgt * dim * 2 > 126e6 else
                   "inputs smaller than L2; the step rewrites >126 MB of operands/candidates between kNN passes")}


DUMP_BYTES = 60 * 10 ** 6     # --dump-outputs stays under 64 MB, .npy headers included


def write_outputs(out_dir, n_rows, records=None, per_row=1, lists=None):
    """--dump-outputs: what a matcher call hands its caller, as out_dir/<name>.npy -- indices and counts in float64 (exact),
    distances and thresholds in float32.  `records`: CORR_DTYPE correspondences of n_rows query rows, ascending index_query,
    at most `per_row` per row; `lists`: the k-lists (idx [n_rows, k], dist [n_rows, k], cnt [n_rows]).  When the largest output
    the workload can produce does not fit DUMP_BYTES, only the outputs of a seeded sample of query rows are written (their
    indices in query_rows.npy).  The sample depends on n_rows and the output shape alone, so every build writes the same rows.
    Returns the names written."""
    row_bytes = 8 + (per_row * 24 if records is not None else lists[0].shape[1] * 12 + 8)   # + 8: query_rows
    rows = None
    if n_rows * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n_rows, DUMP_BYTES // row_bytes, replace=False))
    if records is not None:
        if rows is not None:
            records = records[np.isin(records["index_query"], rows)]
        arrays = {"index_query": records["index_query"].astype(np.float64), "index_match": records["index_match"].astype(np.float64),
                  "distance": records["distance"], "threshold": records["threshold"]}
    else:
        idx, dist, cnt = lists if rows is None else (a[rows] for a in lists)
        arrays = {"knn_index": idx.astype(np.float64), "knn_distance": dist, "knn_count": cnt.astype(np.float64)}
    if rows is not None:
        arrays["query_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
    return sorted(arrays)


# ------------------------------------------------------------------------------------------
def run_b200(args, wl):
    import torch
    import torch.distributed as dist
    from lidar_global_registration_b200 import build as b200_build
    from lidar_global_registration_b200 import device as D
    from lidar_global_registration_b200 import matcher as M
    from lidar_global_registration_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 matcher has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG stays as the caller set it; its log goes to stderr so that stdout carries the ONE JSON line only
        # (the version banner included, whatever NCCL_DEBUG is or defaults to on the box)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        b200_build.build()
    if world > 1:
        dist.barrier()
    be = D.GpuBackend(local_rank)
    sm = D.ShardedMatcher(be, rank, world, None)    # world > 1: attaches the library's own NCCL communicator
    modes = {"mutual": M.MODE_MUTUAL, "ratio": M.MODE_RATIO, "one_sided": M.MODE_ONE_SIDED, "knn_target_sharded": M.MODE_KNN_ONLY}
    pk = peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, sampler=None):
        barrier()
        if sampler:
            sampler.begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    def measure(wl, steps, warmup, with_e2e, with_clocks, dump_dir=None):
        """Device-resident value + candidate-kernel roofline (+ e2e through the host-facing C-ABI) of one workload; with
        dump_dir, the outputs of the last timed step are written there."""
        desc, n_src, n_tgt, k, mode_name, cfg = WORKLOADS[wl]
        tsharded = mode_name == "knn_target_sharded"
        mode = modes[mode_name]
        # target-sharded: every rank generates its own shard of n_tgt rows, global row offset rank * n_tgt
        src, tgt, dim = synth.make_pair_torch(desc, n_src, n_tgt, dev)
        if tsharded and rank > 0:   # a different shard per rank: the common recipe, rows rotated and slightly rescaled
            tgt = (torch.roll(tgt, shifts=1237 * rank, dims=0) * (1.0 + 2e-3 * rank)).contiguous()
        stride_b = src.stride(0) * 4
        t_off = rank * n_tgt if tsharded else 0
        torch.cuda.synchronize()

        def step_device():
            be.upload_device(0, src, dim)
            be.upload_device(1, tgt, dim, index_offset=t_off)
            if tsharded:
                idx, dst, cnt = sm.knn_target_sharded(k)
                return idx, cnt.sum(), dst, cnt
            if world == 1:
                return be.match_device(k, mode)
            return sm.match_query_sharded(k, mode)      # this rank's slice of the records stays in HBM (see config.note)

        # ---- device-resident value (per-kernel CUDA events are recorded on the stream without host syncs) ----
        be.ctx.set_profiling(True)
        sampler = ClockSampler(local_rank) if (rank == 0 and with_clocks) else None
        for _ in range(max(warmup, 3)):
            step_device()
        be.ctx.reset_stats()
        ms_total, out = timed(step_device, steps, sampler)
        clocks = sampler.stop() if sampler else None
        st = be.ctx.stats()
        be.ctx.set_profiling(False)
        n_corr = int(out[1].item())
        res = {"value": n_src * steps / (ms_total * 1e-3), "ms_per_step": ms_total / steps, "launches": int(st["launches"]),
               "clocks": clocks, "dim": dim, "stride_b": stride_b, "n_corr": n_corr}
        if dump_dir:   # copied out before the e2e calls below reuse the context
            if tsharded:
                lists = [x.cpu().numpy() for x in (out[0], out[2], out[3])]
                if rank == 0:
                    write_outputs(dump_dir, n_src, lists=lists)
            else:   # several GPUs: the rank slices in rank order are the single-GPU output
                rec, _ = sm.gather_records(out[0], out[1])
                if rank == 0:
                    write_outputs(dump_dir, n_src, records=rec.cpu().numpy().view(M.CORR_DTYPE).reshape(-1),
                                  per_row=k if mode == M.MODE_MUTUAL else 1)

        # ---- roofline of the dominant kernel (tcgen05 candidate pass): CUDA events around every launch of the timed
        #      region above, on the stream the kernel is launched on ----
        both = mode in (M.MODE_MUTUAL, M.MODE_RATIO_MUTUAL)
        q0, q1 = D.shard_bounds(n_src, rank, world)
        t0, t1 = D.shard_bounds(n_tgt, rank, world)
        pairs_per_step = float((q1 - q0) * n_tgt + ((t1 - t0) * n_src if both else 0))
        if tsharded:   # every rank: all queries against its own target shard
            pairs_per_step = float(n_src) * n_tgt
        # the pairs the candidate kernel actually scored: the masked reverse pass answers only the target rows that forward
        # lists name (st["pairs_scored"] = sum over the launches of rows searched x train rows)
        if st.get("pairs_scored", 0) > 0:
            pairs_per_step = st["pairs_scored"] / steps
        flops_per_step = 2.0 * dim * pairs_per_step
        kpad = (dim + 3 + 15) // 16 * 16           # K the tensor cores actually contract over: D + 3 norm columns, padded to K = 16 steps
        cand_ms = st["ms_candidates"] / steps
        achieved = flops_per_step / (cand_ms * 1e-3) / 1e12 if cand_ms > 0 else 0.0
        n_launch = st["candidate_launches"] / steps
        traffic, traffic_src = ncu_traffic(wl) if world == 1 else (None, None)
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        hw_peak = 148 * 8192.0 * sm_clock * 1e6 / 1e12      # tcgen05 kind::f16: 8192 dense FLOP per SM per cycle
        roofline = {"bound": "tensor", "kernel": "tc_candidates_kernel", "achieved": achieved, "peak": pk["bf16_sustained"],
                    "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"],
                    "peak_source": pk["source"] + ", bf16_tflops_sustained (kernel timed inside a long step; a cuBLAS measurement "
                                   "under the power cap, so a kernel that sustains a higher clock can exceed it)",
                    "frac_of_burst": achieved / pk["bf16_burst"],
                    "frac_of_hw_peak_at_clock": achieved / hw_peak,
                    "hw_peak_at_clock": {"value": hw_peak, "unit": "TFLOP/s", "sm_mhz": sm_clock,
                                         "formula": "148 SMs x 8192 dense FP16 FLOP/cycle/SM x SM clock sampled under load"},
                    "achieved_padded": achieved * kpad / dim,
                    "padded_k": {"k_contracted": kpad, "dim": dim,
                                 "note": "achieved counts 2*D*pairs (SURVEY 8d); the kernel contracts over D + 3 norm columns padded to 16"},
                    "traffic": traffic, "traffic_source": traffic_src,
                    "launch_ms": cand_ms / max(n_launch, 1), "launches_per_step": n_launch,
                    "algorithmic_flops_per_step": flops_per_step,
                    "breakdown_ms_per_step": {x: st[x] / steps for x in ("ms_pack", "ms_prepare", "ms_candidates", "ms_rerank",
                                                                        "ms_fallback", "ms_filter")},
                    # train rows the re-rank scored exactly per query row (FPFH kernels: 32 per surviving chunk entry)
                    "candidates_per_row": st["candidates"] / max(st.get("rows_answered") or st["rows_total"], 1),
                    "query_rows_searched_frac": (st.get("rows_answered") or st["rows_total"]) / max(st["rows_total"], 1),
                    "rows_overflowed_frac": st["rows_flagged"] / max(st["rows_total"], 1)}
        # Second yardstick (SURVEY 8d: for short descriptors the limiter is the accumulator drain + select epilogue, not the
        # tensor pipe): every (query, train) pair's accumulator has to pass the min pipe once.  Measured on this part
        # (tools/ubench/min_ubench.cu): one three-input FMNMX3 (two new values per lane) per 2.25 cycles per scheduler.
        select_peak = 148 * 4 * (64.0 / 2.25) * sm_clock * 1e6
        select_ach = pairs_per_step / (cand_ms * 1e-3) if cand_ms > 0 else 0.0
        roofline["select_epilogue"] = {"achieved": select_ach, "peak": select_peak, "unit": "pairs/s", "frac": select_ach / select_peak,
                                       "peak_source": "148 SMs x 4 schedulers x 64 values per 2.25 cycles (measured FMNMX3 rate) x SM clock under load"}
        res["roofline"] = roofline
        if not with_e2e:
            return res

        # ---- end to end through the host-facing C-ABI: HOST descriptor buffers in, correspondence records on the host out ----
        kk = k if mode == M.MODE_MUTUAL else 1
        src_np, tgt_np = src.cpu().numpy(), tgt.cpu().numpy()              # pageable, as the reference's pcl::PointCloud is
        src_pin, tgt_pin = torch.from_numpy(src_np).pin_memory(), torch.from_numpy(tgt_np).pin_memory()
        e2e = {}
        n_steps = steps
        if world == 1:
            # exactly the calls the C++ shim makes: b200m_upload x 2 + b200m_match (or b200m_knn for the raw k-lists)
            out_np = np.empty(max(n_src * kk, 1), M.CORR_DTYPE)
            for label, (s_h, t_h) in (("pinned", (src_pin.numpy(), tgt_pin.numpy())), ("pageable", (src_np, tgt_np))):
                def step_e2e():
                    be.ctx.upload(0, s_h, dim)
                    be.ctx.upload(1, t_h, dim, index_offset=t_off)
                    if tsharded:
                        r = be.ctx.knn(k, 0)
                        return (r[0].nbytes + r[1].nbytes + r[2].nbytes), None
                    rec, _ = be.ctx.match(k, mode, out=out_np)
                    return rec.shape[0] * 16 + 16, None
                for _ in range(2):
                    step_e2e()
                ms, o = timed(step_e2e, n_steps)
                e2e[label] = {"value": n_src * n_steps / (ms * 1e-3), "ms_per_step": ms / n_steps, "d2h": int(o[0])}
            h2d = src_np.nbytes + tgt_np.nbytes
            res["e2e"] = {"value": e2e["pinned"]["value"], "unit": "queries/s", "h2d_bytes_per_step": int(h2d),
                          "d2h_bytes_per_step": e2e["pinned"]["d2h"], "ms_per_step": e2e["pinned"]["ms_per_step"],
                          "api": "b200m_upload x 2 + b200m_match (the calls include/b200match_shim.hpp makes), pinned host buffers",
                          "pageable_host_buffers": {"value": e2e["pageable"]["value"], "ms_per_step": e2e["pageable"]["ms_per_step"],
                                                    "note": "the same calls from ordinary (pageable) memory, as a pcl::PointCloud is"}}
            return res
        # N > 1: b200m_upload_replicated (1/N slice per rank over PCIe, NVLink all-gather) + b200m_match_sharded -- this rank's
        # slice of the records lands in host memory; the slices in rank order are the single-GPU output
        lists_h = [torch.empty((n_src, k), dtype=torch.int32).pin_memory(), torch.empty((n_src, k), dtype=torch.float32).pin_memory(),
                   torch.empty((n_src,), dtype=torch.int32).pin_memory()] if tsharded else None
        moved = [0, 0]

        def step_e2e_multi():
            if tsharded:   # queries replicated, this rank's own target shard
                moved[0] = sm.upload_host_sharded(0, src_pin, dim) + be.upload_host(1, tgt_pin, dim, index_offset=t_off)
                idx, dst, cnt = sm.knn_target_sharded(k)
                lists_h[0].copy_(idx, non_blocking=True)
                lists_h[1].copy_(dst, non_blocking=True)
                lists_h[2].copy_(cnt, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                moved[1] = (lists_h[0].numel() + lists_h[1].numel() + lists_h[2].numel()) * 4 if rank == 0 else 0
                return None, None
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]   # the library queues on torch's current stream
            ev[0].record()
            moved[0] = sm.upload_host_sharded(0, src_pin, dim)
            ev[1].record()
            moved[0] += sm.upload_host_sharded(1, tgt_pin, dim)
            ev[2].record()
            rec, _ = be.ctx.match_sharded(k, mode)
            ev[3].record()
            phases.append(ev)
            moved[1] = rec.shape[0] * 16 + 16
            return None, None
        phases = []
        for _ in range(2):
            step_e2e_multi()
        del phases[:]
        ms, _ = timed(step_e2e_multi, n_steps)
        tot = torch.tensor(moved, device=dev, dtype=torch.int64)
        dist.all_reduce(tot)
        res["e2e"] = {"value": n_src * n_steps / (ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": int(tot[0].item()),
                      "d2h_bytes_per_step": int(tot[1].item()), "ms_per_step": ms / n_steps,
                      "api": "b200m_upload_replicated x 2 + b200m_match_sharded on every rank (pinned host buffers)",
                      "replication": "each rank copies 1/N of a replicated set over PCIe, NCCL all-gather over NVLink"}
        if phases:
            # where rank 0's end-to-end step goes (CUDA events between the three calls), and what its two transfers cost when
            # nothing else runs: this rank's 1/N slice host -> device, and an all-gather of a replicated set's raw rows
            torch.cuda.synchronize()
            names = ("upload_replicated_src", "upload_replicated_tgt", "match_sharded_incl_result_copy")
            res["e2e"]["rank0_breakdown_ms"] = {nm: sum(p[i].elapsed_time(p[i + 1]) for p in phases) / len(phases) for i, nm in enumerate(names)}
            lo, hi = D.shard_bounds(n_src, rank, world)
            slab = torch.empty((hi - lo, src_pin.shape[1]), dtype=torch.float32, device=dev)
            rows = (n_src + world - 1) // world
            full = torch.empty((rows * world, src_pin.shape[1]), dtype=torch.float32, device=dev)
            part = torch.zeros((rows, src_pin.shape[1]), dtype=torch.float32, device=dev)
            alone = {}
            for nm, fn in (("h2d_slice_alone", lambda: slab.copy_(src_pin[lo:hi], non_blocking=True)),
                           ("allgather_raw_rows_alone", lambda: dist.all_gather_into_tensor(full, part))):
                fn()
                t_ms, _ = timed(fn, 3)
                alone[nm] = t_ms / 3
            res["e2e"]["rank0_breakdown_ms"].update(alone)
        return res

    desc, n_src, n_tgt, k, mode_name, cfg = WORKLOADS[wl]
    tsharded = mode_name == "knn_target_sharded"
    main = measure(wl, args.steps, args.warmup, True, True, args.dump_outputs)

    # the other single-GPU BASELINE configs, embedded so that a default run shows them too (fewer steps, no e2e)
    others = {}
    if wl == "c3" and not args.no_other_configs and (world == 1 or args.other_configs):
        # 1 GPU: the two FPFH configs; several GPUs (only with --other-configs: a collective that fails on one rank must
        # never cost the headline line): the two multi-GPU configs (C4 query-sharded, C5 target-sharded with n_tgt rows per
        # rank -- 8M rows at 8 ranks, BASELINE configs[4])
        for owl, osteps in ((("c2", 10), ("c4", 3)) if world == 1 else (("c4", 3), ("c5", 3))):
            try:
                torch.cuda.empty_cache()
                # an independent workload: it does not inherit the clock state of the one before it (after a second of the
                # SHOT kernel at the 1 kW cap the SM clock stays near 1.5 GHz for a while; a 4 ms FPFH launch measured right
                # behind it runs 10 % slower than on an idle GPU)
                torch.cuda.synchronize()
                time.sleep(3.0)
                o = measure(owl, osteps, 3, False, True)
                od = WORKLOADS[owl]
                others[owl] = {"metric": METRICS[owl], "value": o["value"], "unit": "queries/s", "ms_per_step": o["ms_per_step"],
                               "steps": osteps, "n_gpus": world, "idle_before_s": 3.0, "scaling": "weak" if od[4] == "knn_target_sharded" else "strong",
                               "config": workload_config(owl, world), "correspondences": o["n_corr"],
                               "clocks": o["clocks"], "roofline": o["roofline"],
                               "parity_note": "ratio filter: defined here, the reference's RatioMatcher is a stub (parity unpinned)"
                                              if od[4] == "ratio" else None}
            except Exception as e:   # an embedded extra must never cost the headline line
                others[owl] = {"error": str(e)[:300]}

    # matchLocal with a finite search radius (include/matching.h:637-678) on the C2 shape: cell list vs the gate tested
    # against every train row
    if world == 1 and wl == "c3" and not args.no_other_configs:
        try:
            others["c2_local"] = measure_local(torch, D, M, synth, dev, timed)
        except Exception as e:
            others["c2_local"] = {"error": str(e)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cref = CpuReference(desc, n_src, n_tgt, k, "one_sided" if tsharded else mode_name)
        r, cores, sample, secs = cref.rate(12.0)
        cpu = {"value": r, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample, "seconds": secs,
               "engine": "oracle port of the reference matcher (C, OpenMP)"}
        try:   # beside it: the routine the reference's matchBF calls (OpenCV's BFMatcher through cv2), when cv2 is on the box
            cpu["opencv_bfmatcher"] = opencv_bfmatcher_rate(cref, 5.0)
        except Exception as e:
            cpu["opencv_bfmatcher"] = {"error": str(e)[:200]}

    if rank == 0:
        note = None
        if world > 1 and not tsharded:
            note = ("the timed step leaves every rank's slice of the records in its own HBM (ascending index_query; the slices in "
                    "rank order are the single-GPU output); gathering them to one rank (8 MB for c3) is outside the timed region")
        line = {"metric": METRICS[wl], "value": main["value"], "unit": "queries/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": main["ms_per_step"], "higher_is_better": True,
                "scaling": "weak" if tsharded else "strong", "vs_baseline": None,
                "dtype": "f32 (FP16 tensor-core candidates, exact FP32 re-rank)",
                "data": "synthetic",
                "config": workload_config(wl, world), "correspondences": main["n_corr"], "note": note,
                "e2e": main["e2e"], "gpu_launches": main["launches"], "clocks": main["clocks"], "roofline": main["roofline"],
                "cpu_baseline": cpu, "other_configs": others or None}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    be.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the embedded c2 / c4 lines of a default (c3, 1 GPU) run")
    ap.add_argument("--other-configs", action="store_true", help="several GPUs: also embed the c4 (query-sharded) and c5 (target-sharded) lines")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs (the reference arm times a sample sized by the clock)")
    # stdout carries the ONE JSON line and nothing else: whatever a library prints through C stdio or fd 1 during the run
    # (NCCL's "NCCL version ..." banner does, on boxes where NCCL_DEBUG defaults to VERSION, NCCL_DEBUG_FILE or not) goes to
    # stderr; the line itself is written to the saved descriptor at the end.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            if args.impl == "reference":
                run_reference(args, args.workload)
            else:
                run_b200(args, args.workload)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    lines = [ln for ln in buf.getvalue().splitlines() if ln.strip()]
    for ln in lines[:-1]:            # anything python printed besides the line: to stderr
        sys.stderr.write(ln + "\n")
    if lines:
        sys.stdout.write(lines[-1] + "\n")
        sys.stdout.flush()


if __name__ == "__main__":
    main()
