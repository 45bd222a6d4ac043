"""Loop of single-pair calls vs one batch call, on the same seeded pinned host inputs.  Prints one JSON line.

    python tools/bench_batch.py [--reps N] [--out FILE]

Arms (alternated in one run, after a warm-up of each; host clock around calls that end in a device synchronise):
    loop   per pair b200m_upload(0) + b200m_upload(1) + b200m_match -- what a caller does today, one pair per call
    batch  one b200m_match_batch over all pairs
Workloads: FPFH-33 20k x 20k, k = 1, mutual (BASELINE's C1 shape) for B in {1, 16, 64, 256}; SHOT-352 5k x 5k, k = 2, mutual
for B in {1, 64}.  Distinct seeded pairs (at most 64 per workload, repeated cyclically beyond); the arms' records and averages
are asserted identical.  A separate profiled batch call gives the b200m_get_stats breakdown; the candidate kernel's
algorithmic rate is 2 * dim * (forward + reverse (query, train) pairs of all pairs) over its launch time.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from lidar_global_registration_b200 import matcher as M   # noqa: E402
from lidar_global_registration_b200 import synth           # noqa: E402

WORKLOADS = [("fpfh", 20000, 1, [1, 16, 64, 256]), ("shot", 5000, 2, [1, 64])]
MAX_DISTINCT = 64


def pinned_pairs(desc, n, count):
    import torch
    out = []
    for i in range(min(count, MAX_DISTINCT)):
        s, t, dim = synth.make_pair(desc, n, n, seed=1000 + i, nan_frac=0.001)
        ps = torch.empty(s.shape, dtype=torch.float32, pin_memory=True).numpy()
        pt = torch.empty(t.shape, dtype=torch.float32, pin_memory=True).numpy()
        ps[...] = s
        pt[...] = t
        out.append((ps, pt))
    return [out[i % len(out)] for i in range(count)], dim


def run_loop(ctx, pairs, dim, k, mode):
    L, h = ctx._L, ctx._h
    p = M.Context._params(k, mode)
    res = []
    for s, t in pairs:
        stride = s.strides[0]
        ctx._ck(L.b200m_upload(h, 0, s.ctypes.data, s.shape[0], stride, dim, 0))
        ctx._ck(L.b200m_upload(h, 1, t.ctypes.data, t.shape[0], stride, dim, 0))
        out = np.empty(s.shape[0] * (k if mode == M.MODE_MUTUAL else 1), M.CORR_DTYPE)
        n, avg = C.c_size_t(0), C.c_float(0)
        ctx._ck(L.b200m_match(h, C.byref(p), None, None, out.ctypes.data, out.shape[0], C.byref(n), C.byref(avg)))
        res.append((out[:n.value], avg.value))
    return res


def run_batch(ctx, pairs, dim, k, mode, arr, stride):
    L, h = ctx._L, ctx._h
    p = M.Context._params(k, mode)
    out = np.empty(sum(s.shape[0] for s, _ in pairs) * (k if mode == M.MODE_MUTUAL else 1), M.CORR_DTYPE)
    offsets = np.zeros(len(pairs) + 1, np.uint64)
    avg = np.empty(len(pairs), np.float32)
    ctx._ck(L.b200m_match_batch(h, C.byref(p), arr, len(pairs), stride, dim, None, None, out.ctypes.data, out.shape[0],
                                offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data))
    return [(out[int(offsets[i]):int(offsets[i + 1])], float(avg[i])) for i in range(len(pairs))]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    mode = M.MODE_MUTUAL
    name, power = card()
    rows = []
    with M.Context(0) as ctx:
        for desc, n, k, batches in WORKLOADS:
            all_pairs, dim = pinned_pairs(desc, n, max(batches))
            for B in batches:
                pairs = all_pairs[:B]
                keep, arr, stride, _ = M.Context._pairs(pairs, dim)
                ref = run_loop(ctx, pairs, dim, k, mode)                       # warm-up of both arms
                got = run_batch(ctx, pairs, dim, k, mode, arr, stride)
                for (r0, a0), (r1, a1) in zip(ref, got):
                    assert r0.tobytes() == r1.tobytes() and np.float32(a0) == np.float32(a1), "loop and batch differ"
                t_loop, t_batch = [], []
                for _ in range(a.reps):
                    t = time.perf_counter()
                    run_loop(ctx, pairs, dim, k, mode)
                    t_loop.append(time.perf_counter() - t)
                    t = time.perf_counter()
                    run_batch(ctx, pairs, dim, k, mode, arr, stride)
                    t_batch.append(time.perf_counter() - t)
                ctx.set_profiling(True)
                ctx.reset_stats()
                run_batch(ctx, pairs, dim, k, mode, arr, stride)
                st = ctx.stats()
                ctx.set_profiling(False)
                ml, mb = statistics.median(t_loop), statistics.median(t_batch)
                scored = 2 * sum(s.shape[0] * t.shape[0] for s, t in pairs)   # forward + reverse (mutual)
                queries = sum(s.shape[0] for s, _ in pairs)
                rows.append({
                    "workload": "%s-%d %dx%d k=%d mutual" % (desc, dim, n, n, k), "pairs": B,
                    "distinct_pairs": min(B, MAX_DISTINCT),
                    "loop_ms": round(ml * 1e3, 3), "batch_ms": round(mb * 1e3, 3), "speedup": round(ml / mb, 2),
                    "loop_pairs_per_s": round(B / ml, 1), "batch_pairs_per_s": round(B / mb, 1),
                    "loop_queries_per_s": round(queries / ml), "batch_queries_per_s": round(queries / mb),
                    "loop_ms_all": [round(x * 1e3, 3) for x in t_loop], "batch_ms_all": [round(x * 1e3, 3) for x in t_batch],
                    "batch_stats": {kk: (round(v, 4) if isinstance(v, float) else v) for kk, v in st.items()},
                    "candidate_tflops": round(2.0 * dim * scored / (st["ms_candidates"] * 1e-3) / 1e12, 1)
                    if st["ms_candidates"] > 0 else None,
                })
                print("%-28s B=%-3d loop %8.2f ms  batch %8.2f ms  x%.2f" % (rows[-1]["workload"], B, ml * 1e3, mb * 1e3, ml / mb),
                      file=sys.stderr)
    line = json.dumps({"tool": "bench_batch", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
