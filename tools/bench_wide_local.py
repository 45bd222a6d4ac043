"""Loop of one-pair b200m_match_multiscale_local_batch calls vs one call over all pairs (the matcher classes with
AlignmentParameters::guess set), on the same seeded inputs.  Prints one JSON line.

    python tools/bench_wide_local.py [--reps N] [--out FILE]

Arms (alternated in one run, after a warm-up of each; host clock around calls that end in a device synchronise; both go
through Context.match_wide_local_batch, so both include its Python argument marshalling):
    loop   per pair one call with that pair alone -- what FeatureBasedMatcher.match() does with a guess
    batch  one call over all pairs -- what match_many does
Workloads (keypoints uniform in a 40 m cube with a quarter in one 0.2 m cluster; a small rigid guess per pair):
    LeftToRightMatcher  FPFH-33, 20k keypoints, 3 scales (20k, 16k, 12k rows), k = 2, radius 4.7 (about 10^2 gated rows
                        per query), B in {16, 64}
    ClusterMatcher      SHOT-352, 5k keypoints, 2 scales (5k, 4k rows), k = 2, radius 4.7, B = 64
    ClusterMatcher      FPFH-33, 5k keypoints, 1 scale, k = 1, radius FLT_MAX (every row passes: one cell per grid), B = 16
The arms' records and averages are asserted identical.  b200m_get_stats gives the launches per call of both arms; a
torch.profiler pass over one batch call, in its own run, gives the gated kNN's share of kernel time.
"""
import argparse
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

# (name, mode, descriptor, keypoints, rows per scale as a fraction of the keypoints, k, radius, batch sizes)
WORKLOADS = [("lr fpfh 20k 3 scales", M.MODE_MUTUAL, "fpfh", 20000, [1.0, 0.8, 0.6], 2, 4.7, [16, 64]),
             ("cluster shot 5k 2 scales", M.MODE_CLUSTER, "shot", 5000, [1.0, 0.8], 2, 4.7, [64]),
             ("cluster fpfh 5k whole-cloud radius", M.MODE_CLUSTER, "fpfh", 5000, [1.0], 1, M.FLT_MAX, [16])]
MAX_DISTINCT = 16


def rigid(rng, angle=0.05, shift=0.5):
    ax = rng.standard_normal(3)
    ax /= np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    t = angle * rng.random()
    g = np.eye(4)
    g[:3, :3] = np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K
    g[:3, 3] = shift * rng.standard_normal(3)
    return g.astype(np.float32)


def make_pairs(desc, n, fracs, count):
    pairs, dim = [], None
    for i in range(min(count, MAX_DISTINCT)):
        rng = np.random.default_rng(700 + i)
        xyz = []
        for _ in range(2):
            x = np.zeros((n, 4), np.float32)
            x[:, :3] = rng.random((n, 3)) * 40
            x[: n // 4, :3] = x[0, :3] + 0.2 * rng.standard_normal((n // 4, 3)).astype(np.float32)
            xyz.append(x)
        s_sc, t_sc = [], []
        for s, f in enumerate(fracs):
            m = int(n * f)
            src, tgt, dim = synth.make_pair(desc, m, m, seed=3000 + 10 * i + s, nan_frac=0.001)
            maps = [None if m == n else np.sort(rng.choice(n, m, replace=False)).astype(np.int32) for _ in range(2)]
            s_sc.append((src, maps[0]))
            t_sc.append((tgt, maps[1]))
        g = rigid(rng)
        pairs.append(dict(src_scales=s_sc, tgt_scales=t_sc, src_kps_xyz=xyz[0], tgt_kps_xyz=xyz[1],
                          iss_radius_src=0.3 + 0.1 * rng.random(), iss_radius_tgt=0.3 + 0.1 * rng.random(),
                          src_kps_moved=M.transform_keypoints(xyz[0], g), tgt_kps_moved=M.transform_keypoints(xyz[1], M.invert_guess(g))))
    return [pairs[i % len(pairs)] for i in range(count)], dim


def launches(ctx, fn):
    ctx.reset_stats()
    fn()
    return ctx.stats()["launches"]


GATED = ("seg_gather", "seg_bbox", "seg_grid", "cell_count", "cell_scan", "cell_fill", "local_cells")


def kernel_shares(fn):
    """torch.profiler over one call: device time per kernel group (ms) and the gated kNN's share of all kernel time"""
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
            key = next((w for w in GATED + ("knn3d", "ms_vote", "ms_scatter_batch", "cluster_dist", "pack", "filter", "average",
                                            "localize") if w in e.key), "other")
            per[key] = per.get(key, 0.0) + t / 1e3
    total = sum(per.values())
    gated = sum(v for k, v in per.items() if k in GATED)
    return {"kernel_ms_total": round(total, 3), "kernel_ms": {k: round(v, 3) for k, v in sorted(per.items(), key=lambda x: -x[1])},
            "gated_knn_share": round(gated / total, 4) if total else None}


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
        for wname, mode, desc, n, fracs, k, radius, batches in WORKLOADS:
            all_pairs, dim = make_pairs(desc, n, fracs, max(batches))
            for B in batches:
                pairs = all_pairs[:B]
                loop = lambda: [ctx.match_wide_local_batch(k, mode, [pr], radius, dim)[0] for pr in pairs]   # noqa: E731
                batch = lambda: ctx.match_wide_local_batch(k, mode, pairs, radius, dim)                      # noqa: E731
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
                shares = kernel_shares(batch)
                ml, mb = statistics.median(t_loop), statistics.median(t_batch)
                rows.append({
                    "workload": wname, "mode": mode, "k": k, "keypoints": n, "scales": len(fracs), "radius": radius, "pairs": B,
                    "distinct_pairs": min(B, MAX_DISTINCT), "records": sum(len(r) for r, _ in got),
                    "loop_ms": round(ml * 1e3, 3), "batch_ms": round(mb * 1e3, 3), "loop_over_batch": round(ml / mb, 2),
                    "loop_ms_all": [round(x * 1e3, 3) for x in t_loop], "batch_ms_all": [round(x * 1e3, 3) for x in t_batch],
                    "loop_launches": n_loop, "batch_launches": n_batch, "batch_kernels": shares,
                })
                print("%-36s B=%-3d loop %9.2f ms  batch %9.2f ms  x%.2f  launches %d / %d  gated %s" % (
                    wname, B, ml * 1e3, mb * 1e3, ml / mb, n_loop, n_batch, shares["gated_knn_share"]), file=sys.stderr)
    line = json.dumps({"tool": "bench_wide_local", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
