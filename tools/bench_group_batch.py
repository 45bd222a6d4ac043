"""Host batch calls on one context vs the same calls on a b200m_group (the pairs spread over 1, 2, 4, 8 GPUs, as many as
the box has), on the same seeded pageable host inputs.  Prints one JSON line.

    python tools/bench_group_batch.py [--reps N] [--out FILE]

Arms (alternated in one run, after a warm-up of each; host clock around calls that end in a device synchronise):
    single   b200m_match_batch / b200m_match_multiscale(_local)_batch on one context (GPU 0)
    group-W  b200m_group_* on a group of the first W GPUs
Workloads:
    match batch      FPFH-33 20k x 20k, k = 1, mutual, B = 64 and 256
    LeftToRight      FPFH-33 20k keypoints, 3 scales (20k, 16k, 12k rows), k = 2, B = 64
    ClusterMatcher   SHOT-352 5k keypoints, 2 scales, k = 2, B = 64
    ClusterMatcher   FPFH-33 20k keypoints, 1 scale, k = 1, B = 64 (bound by the 3-D neighbourhoods, knn3d)
    LeftToRight      the same pair with k = 1, 1 scale, B = 64: with the ClusterMatcher row above it sets the knn3d constant
                     of the cost model (c3d = (T_cluster - T_lr) / T_lr * desc_cost / knn3d pairs)
    guessed LR       FPFH-33 20k keypoints, 3 scales, k = 2, match_search_radius 4.7, B = 64
Distinct seeded pairs (16 per workload, repeated cyclically beyond, as tools/bench_wide_batch.py makes them); every arm's
records, offsets and averages are asserted identical to the single arm's.  Per group device the profiled stage time of one
call (b200m_get_stats on b200m_group_ctx(g, i) with profiling on, a separate untimed call) shows how even the split is.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from lidar_global_registration_b200 import matcher as M   # noqa: E402
from lidar_global_registration_b200 import synth           # noqa: E402
import bench_wide_batch as BW                              # noqa: E402

BW.pinned = lambda a: a   # pageable host memory, as a caller's numpy arrays are

RADIUS = 4.7
GUESS = (0.9950042, -0.0998334, 0.0, 0.3, 0.0998334, 0.9950042, 0.0, -0.2, 0.0, 0.0, 1.0, 0.1, 0.0, 0.0, 0.0, 1.0)
STAGES = ("ms_pack", "ms_prepare", "ms_candidates", "ms_rerank", "ms_fallback", "ms_filter")


def narrow_workload(B):
    pairs = []
    for i in range(min(B, 16)):
        s, t, dim = synth.make_pair("fpfh", 20000, 20000, seed=700 + i, nan_frac=0.001)
        pairs.append((s, t))
    pairs = [pairs[i % len(pairs)] for i in range(B)]
    arr = (M._Pair * B)()
    for i, (s, t) in enumerate(pairs):
        arr[i] = M._Pair(s.ctypes.data, s.shape[0], t.ctypes.data, t.shape[0])
    n_src = sum(s.shape[0] for s, _ in pairs)
    stride = pairs[0][0].strides[0]

    def call(target, fn, keep=pairs):   # keep: the descriptor arrays `arr` points into live as long as the call
        out = np.empty(n_src, M.CORR_DTYPE)
        offsets = np.zeros(B + 1, np.uint64)
        avg = np.empty(B, np.float32)
        p = M.Context._params(1, M.MODE_MUTUAL)
        target._ck(fn(target._h, C.byref(p), arr, B, stride, dim, None, None, out.ctypes.data, out.shape[0],
                      offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data))
        return out[:int(offsets[-1])].tobytes() + offsets.tobytes() + avg.tobytes()
    return call, "match_batch"


def desc_cost(nq, nt, dim):
    return nq * nt * ((dim + 3 + 63) // 64 * 64)


def wide_workload(desc, n, fracs, k, mode, B, guessed=False):
    pairs = BW.make_pairs(desc, n, fracs, B)
    arrs = [BW.scale_array(pr) for pr in pairs]
    wide = (M._WidePair * B)()
    locs = (M._LocalPair * B)()
    keep = [pairs, arrs]
    for i, (pr, arr) in enumerate(zip(pairs, arrs)):
        sx, tx = pr["xyz"]
        wide[i] = M._WidePair(C.cast(arr, C.c_void_p), len(pr["scales"]), sx.ctypes.data, sx.shape[0], tx.ctypes.data, tx.shape[0],
                              pr["iss"][0], pr["iss"][1])
        if guessed:
            ms, mt = M.transform_keypoints(sx, GUESS), M.transform_keypoints(tx, M.invert_guess(GUESS))
            keep += [ms, mt]
            locs[i] = M._LocalPair(ms.ctypes.data, mt.ctypes.data)
    n_src = sum(pr["xyz"][0].shape[0] for pr in pairs)
    src, sx = pairs[0]["scales"][0][0], pairs[0]["xyz"][0]
    dim = pairs[0]["dim"]

    def call(target, fn, keep=keep):   # keep: every array `wide` and `locs` point into lives as long as the call
        out = np.empty(n_src, M.CORR_DTYPE)
        offsets = np.zeros(B + 1, np.uint64)
        avg = np.empty(B, np.float32)
        p = M.Context._params(k, mode)
        tail = (None, None, out.ctypes.data, out.shape[0], offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data)
        if guessed:
            target._ck(fn(target._h, C.byref(p), wide, locs, B, src.strides[0], dim, sx.strides[0], 40, RADIUS, *tail))
        else:
            target._ck(fn(target._h, C.byref(p), wide, B, src.strides[0], dim, sx.strides[0], 40, *tail))
        return out[:int(offsets[-1])].tobytes() + offsets.tobytes() + avg.tobytes()
    return call, "match_multiscale_local_batch" if guessed else "match_multiscale_batch"


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = BW.card()
    n_dev = torch.cuda.device_count()
    widths = [w for w in (1, 2, 4, 8) if w <= n_dev]
    workloads = [
        ("match fpfh 20k k=1 mutual", lambda: narrow_workload(64), 64),
        ("match fpfh 20k k=1 mutual", lambda: narrow_workload(256), 256),
        ("lr fpfh 20k 3 scales k=2", lambda: wide_workload("fpfh", 20000, [1.0, 0.8, 0.6], 2, M.MODE_MUTUAL, 64), 64),
        ("cluster shot 5k 2 scales k=2", lambda: wide_workload("shot", 5000, [1.0, 0.8], 2, M.MODE_CLUSTER, 64), 64),
        ("cluster fpfh 20k 1 scale k=1", lambda: wide_workload("fpfh", 20000, [1.0], 1, M.MODE_CLUSTER, 64), 64),
        ("lr fpfh 20k 1 scale k=1", lambda: wide_workload("fpfh", 20000, [1.0], 1, M.MODE_MUTUAL, 64), 64),
        ("guessed lr fpfh 20k 3 scales k=2 r=4.7", lambda: wide_workload("fpfh", 20000, [1.0, 0.8, 0.6], 2, M.MODE_MUTUAL, 64,
                                                                          guessed=True), 64),
    ]
    rows = []
    ctx = M.Context(0)
    groups = {w: M.Group(list(range(w))) for w in widths}
    try:
        for wname, make, B in workloads:
            call, fn = make()
            arms = {"single": lambda: call(ctx, getattr(ctx._L, "b200m_" + fn))}
            for w, g in groups.items():
                arms["group-%d" % w] = (lambda g=g: call(g, getattr(g._L, "b200m_group_" + fn)))
            ref = arms["single"]()
            for arm, f in arms.items():   # warm-up, and the outputs of every arm equal the single context's
                assert f() == ref, (wname, arm)
            times = {arm: [] for arm in arms}
            for _ in range(a.reps):
                for arm, f in arms.items():
                    t = time.perf_counter()
                    f()
                    times[arm].append(time.perf_counter() - t)
            med = {arm: statistics.median(v) * 1e3 for arm, v in times.items()}
            per_dev = {}
            for w, g in groups.items():
                L = g._L
                for i in range(w):
                    L.b200m_set_profiling(L.b200m_group_ctx(g._h, i), 1)
                    L.b200m_reset_stats(L.b200m_group_ctx(g._h, i))
                arms["group-%d" % w]()
                busy = []
                for i in range(w):
                    h = L.b200m_group_ctx(g._h, i)
                    st = M.Stats()
                    L.b200m_get_stats(h, C.byref(st))
                    busy.append(round(sum(getattr(st, s) for s in STAGES), 3))
                    L.b200m_set_profiling(h, 0)
                per_dev["group-%d" % w] = busy
            row = {"workload": wname, "pairs": B, "ms": {k: round(v, 3) for k, v in med.items()},
                   "ms_all": {k: [round(x * 1e3, 3) for x in v] for k, v in times.items()},
                   "speedup_vs_single": {k: round(med["single"] / v, 3) for k, v in med.items()},
                   "efficiency": {"group-%d" % w: round(med["group-1"] / (w * med["group-%d" % w]), 3) for w in widths},
                   "profiled_stage_ms_per_device": per_dev, "records_bytes": len(ref)}
            rows.append(row)
            print("%-40s B=%-3d %s" % (wname, B, "  ".join("%s %.2f ms" % (k, v) for k, v in med.items())), file=sys.stderr)
        cl = next(r for r in rows if r["workload"].startswith("cluster fpfh 20k"))["ms"]["group-1"]
        lr = next(r for r in rows if r["workload"].startswith("lr fpfh 20k 1 scale"))["ms"]["group-1"]
        # per pair: desc_cost = 2 directions x 20k x 20k x 64, knn3d = 2 x 20k^2 keypoint pairs
        c3d = (cl - lr) / lr * (2 * desc_cost(20000, 20000, 33)) / (2 * 20000.0 ** 2)
    finally:
        for g in groups.values():
            g.close()
        ctx.close()
    line = json.dumps({"tool": "bench_group_batch", "gpu": name, "power_limit": power, "devices": n_dev, "reps": a.reps,
                       "c3d_measured": round(c3d, 1), "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
