"""Loop of single-pair b200m_match_multiscale calls vs one b200m_match_multiscale_batch call, on the same seeded pinned
host inputs.  Prints one JSON line.

    python tools/bench_wide_batch.py [--reps N] [--out FILE]

Arms (alternated in one run, after a warm-up of each; host clock around calls that end in a device synchronise):
    loop   per pair one b200m_match_multiscale -- what a caller of the matcher classes does today, one pair per call
    batch  one b200m_match_multiscale_batch over all pairs
Workloads (the matcher classes at the wide seam):
    ClusterMatcher      FPFH-33, 20k x 20k keypoints, 1 scale, k = 1, B in {1, 16, 64}
    LeftToRightMatcher  FPFH-33, 3 scales (20k, 16k, 12k rows with index maps), k = 2, B in {1, 16}
    ClusterMatcher      SHOT-352, 5k x 5k keypoints, 2 scales (5k, 4k rows), k = 2, B = 64
Distinct seeded pairs (at most 16 per workload, repeated cyclically beyond); the arms' records and averages are asserted
identical.  b200m_get_stats gives the launches per call of both arms and, in a profiled batch call, the time per stage;
a torch.profiler pass over one batch call gives the kernel-time share of the 3-D neighbourhoods (knn3d) and the others.
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

# (name, mode, descriptor, keypoints, rows per scale as a fraction of the keypoints, k, batch sizes)
WORKLOADS = [("cluster fpfh 20k 1 scale", M.MODE_CLUSTER, "fpfh", 20000, [1.0], 1, [1, 16, 64]),
             ("lr fpfh 20k 3 scales", M.MODE_MUTUAL, "fpfh", 20000, [1.0, 0.8, 0.6], 2, [1, 16]),
             ("cluster shot 5k 2 scales", M.MODE_CLUSTER, "shot", 5000, [1.0, 0.8], 2, [64])]
MAX_DISTINCT = 16


def pinned(a):
    import torch
    out = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True).numpy()
    out[...] = a
    return out


def make_pairs(desc, n, fracs, count):
    """one pair = dict of pinned arrays: per scale (src rows, src map, tgt rows, tgt map), keypoints, radii"""
    pairs = []
    for i in range(min(count, MAX_DISTINCT)):
        rng = np.random.default_rng(500 + i)
        xyz = []
        for _ in range(2):
            x = np.zeros((n, 4), np.float32)
            x[:, :3] = rng.random((n, 3)) * 40
            x[: n // 4, :3] = x[0, :3] + 0.2 * rng.standard_normal((n // 4, 3)).astype(np.float32)
            xyz.append(pinned(x))
        scales = []
        for s, f in enumerate(fracs):
            m = int(n * f)
            src, tgt, dim = synth.make_pair(desc, m, m, seed=2000 + 10 * i + s, nan_frac=0.001)
            maps = [None if m == n else pinned(np.sort(rng.choice(n, m, replace=False)).astype(np.int32)) for _ in range(2)]
            scales.append((pinned(src), maps[0], pinned(tgt), maps[1]))
        pairs.append({"scales": scales, "xyz": xyz, "iss": (0.3 + 0.1 * rng.random(), 0.3 + 0.1 * rng.random()), "dim": dim})
    return [pairs[i % len(pairs)] for i in range(count)]


def scale_array(pr):
    arr = (M._Scale * len(pr["scales"]))()
    for s, (src, smap, tgt, tmap) in enumerate(pr["scales"]):
        arr[s] = M._Scale(src.ctypes.data, src.shape[0], None if smap is None else smap.ctypes.data, tgt.ctypes.data, tgt.shape[0],
                          None if tmap is None else tmap.ctypes.data)
    return arr


def run_loop(ctx, pairs, arrs, k, mode):
    L, h = ctx._L, ctx._h
    p = M.Context._params(k, mode)
    res = []
    for pr, arr in zip(pairs, arrs):
        src = pr["scales"][0][0]
        sx, tx = pr["xyz"]
        out = np.empty(sx.shape[0], M.CORR_DTYPE)
        n, avg = C.c_size_t(0), C.c_float(0)
        ctx._ck(L.b200m_match_multiscale(h, C.byref(p), arr, len(pr["scales"]), src.strides[0], pr["dim"], sx.ctypes.data,
                                         sx.shape[0], tx.ctypes.data, tx.shape[0], sx.strides[0], pr["iss"][0], pr["iss"][1], 40,
                                         None, None, out.ctypes.data, out.shape[0], C.byref(n), C.byref(avg)))
        res.append((out[:n.value], avg.value))
    return res


def run_batch(ctx, pairs, wide, k, mode):
    L, h = ctx._L, ctx._h
    p = M.Context._params(k, mode)
    src, sx = pairs[0]["scales"][0][0], pairs[0]["xyz"][0]
    out = np.empty(sum(pr["xyz"][0].shape[0] for pr in pairs), M.CORR_DTYPE)
    offsets = np.zeros(len(pairs) + 1, np.uint64)
    avg = np.empty(len(pairs), np.float32)
    ctx._ck(L.b200m_match_multiscale_batch(h, C.byref(p), wide, len(pairs), src.strides[0], pairs[0]["dim"], sx.strides[0], 40,
                                           None, None, out.ctypes.data, out.shape[0],
                                           offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data))
    return [(out[int(offsets[i]):int(offsets[i + 1])], float(avg[i])) for i in range(len(pairs))]


def launches(ctx, fn):
    ctx.reset_stats()
    fn()
    return ctx.stats()["launches"]


def kernel_shares(ctx, fn):
    """torch.profiler over one call: device time per kernel name (ms) and the knn3d share of all kernel time"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0)
        if t > 0 and not e.key.startswith("Memcpy") and not e.key.startswith("Memset"):
            per[e.key] = per.get(e.key, 0.0) + t / 1e3
    total = sum(per.values())
    short = {}
    for name, ms in per.items():
        key = next((w for w in ("knn3d", "ms_vote", "ms_scatter_batch", "cluster_dist", "candidates", "rerank", "exact", "pack",
                                "filter", "average", "localize") if w in name), "other")
        short[key] = short.get(key, 0.0) + ms
    return {"kernel_ms_total": round(total, 3), "kernel_ms": {k: round(v, 3) for k, v in sorted(short.items(), key=lambda x: -x[1])},
            "knn3d_share": round(short.get("knn3d", 0.0) / total, 4) if total else None}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    rows = []
    with M.Context(0) as ctx:
        for wname, mode, desc, n, fracs, k, batches in WORKLOADS:
            all_pairs = make_pairs(desc, n, fracs, max(batches))
            for B in batches:
                pairs = all_pairs[:B]
                arrs = [scale_array(pr) for pr in pairs]
                wide = (M._WidePair * B)()
                for i, (pr, arr) in enumerate(zip(pairs, arrs)):
                    sx, tx = pr["xyz"]
                    wide[i] = M._WidePair(C.cast(arr, C.c_void_p), len(pr["scales"]), sx.ctypes.data, sx.shape[0], tx.ctypes.data,
                                          tx.shape[0], pr["iss"][0], pr["iss"][1])
                loop = lambda: run_loop(ctx, pairs, arrs, k, mode)        # noqa: E731
                batch = lambda: run_batch(ctx, pairs, wide, k, mode)       # noqa: E731
                ref, got = loop(), batch()                                 # warm-up of both arms
                for (r0, a0), (r1, a1) in zip(ref, got):
                    assert r0.tobytes() == r1.tobytes() and np.float32(a0) == np.float32(a1), "loop and batch differ"
                t_loop, t_batch = [], []
                for _ in range(a.reps):
                    t = time.perf_counter()
                    loop()
                    t_loop.append(time.perf_counter() - t)
                    t = time.perf_counter()
                    batch()
                    t_batch.append(time.perf_counter() - t)
                n_loop, n_batch = launches(ctx, loop), launches(ctx, batch)
                ctx.set_profiling(True)
                ctx.reset_stats()
                batch()
                st = ctx.stats()
                ctx.set_profiling(False)
                shares = kernel_shares(ctx, batch)
                ml, mb = statistics.median(t_loop), statistics.median(t_batch)
                rows.append({
                    "workload": wname, "mode": mode, "k": k, "keypoints": n, "scales": len(fracs), "pairs": B,
                    "distinct_pairs": min(B, MAX_DISTINCT), "records": sum(len(r) for r, _ in got),
                    "loop_ms": round(ml * 1e3, 3), "batch_ms": round(mb * 1e3, 3), "speedup": round(ml / mb, 2),
                    "loop_ms_all": [round(x * 1e3, 3) for x in t_loop], "batch_ms_all": [round(x * 1e3, 3) for x in t_batch],
                    "loop_launches": n_loop, "batch_launches": n_batch,
                    "batch_stats": {kk: (round(v, 4) if isinstance(v, float) else v) for kk, v in st.items()},
                    "batch_kernels": shares,
                })
                print("%-26s B=%-3d loop %8.2f ms  batch %8.2f ms  x%.2f  launches %d / %d  knn3d %s" % (
                    wname, B, ml * 1e3, mb * 1e3, ml / mb, n_loop, n_batch, shares["knn3d_share"]), file=sys.stderr)
    line = json.dumps({"tool": "bench_wide_batch", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
