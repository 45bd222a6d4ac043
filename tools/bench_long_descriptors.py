"""Long descriptors (kp > 640) on the K-streamed tensor-core pass against the exact CUDA-core path, on the same seeded
inputs.  Prints one JSON line.

    python tools/bench_long_descriptors.py [--reps N] [--out FILE] [--only NAME]

Timing: host clock around calls that end in a device synchronise (Context.match returns host records), median of N
alternated repetitions after a warm-up of every arm; outputs are asserted identical between the arms.  One more call per
arm with profiling on gives b200m_get_stats: the candidate kernel's time, candidates per row, flagged rows and the re-rank
time.  TFLOP/s is algorithmic: 2 * D * (query rows searched x train rows) over the candidate kernel's time, the pairs
counted by b200m_get_stats (the masked reverse pass of a mutual match searches only the target rows the forward lists name).
Workloads:
    usc 20k       USC-1960 20k x 20k, k = 1, mutual: default against F32_EXACT (the only GPU route for rows this long before)
    usc 100k      USC-1960 100k x 100k, k = 2, mutual, tensor-core path only (operands 400 MB per side, beyond the 126 MB of
                  L2), 256 sampled rows checked against the oracle
    dim 700 50k / dim 1024 50k   50k x 50k, k = 1, mutual: the first 700 / 1024 columns of USC-like rows, default against exact
    cluster usc   ClusterMatcher, USC-1960 5k keypoints, 2 scales (5k, 4k rows), k = 2, 16 pairs in one match_wide_batch
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
from oracle import oracle as orc                           # noqa: E402

PEAK_TFLOPS = 1388.0   # sustained FP16 dense rate DESIGN.md quotes for one B200 at a 1000 W power limit


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def usc_rows(n_src, n_tgt, seed, dim=None):
    import torch
    s, t, d = synth.make_pair_torch("usc", n_src, n_tgt, "cuda:0", seed=seed)
    dim = dim or d
    out = (np.ascontiguousarray(s[:, :dim].cpu().numpy()), np.ascontiguousarray(t[:, :dim].cpu().numpy()), dim) \
        if dim != d else (s.cpu().numpy(), t.cpu().numpy(), d)
    del s, t
    torch.cuda.empty_cache()
    return out


def wide_pairs(n, fracs, count):
    pairs, dim = [], None
    for i in range(count):
        rng = np.random.default_rng(900 + i)
        xyz = []
        for _ in range(2):
            x = np.zeros((n, 4), np.float32)
            x[:, :3] = rng.random((n, 3)) * 40
            x[: n // 4, :3] = x[0, :3] + 0.2 * rng.standard_normal((n // 4, 3)).astype(np.float32)
            xyz.append(x)
        s_sc, t_sc = [], []
        for s, f in enumerate(fracs):
            m = int(n * f)
            src, tgt, dim = synth.make_pair("usc", m, m, seed=6000 + 10 * i + s, nan_frac=0.001)
            maps = [None if m == n else np.sort(rng.choice(n, m, replace=False)).astype(np.int32) for _ in range(2)]
            s_sc.append((src, maps[0]))
            t_sc.append((tgt, maps[1]))
        pairs.append(dict(src_scales=s_sc, tgt_scales=t_sc, src_kps_xyz=xyz[0], tgt_kps_xyz=xyz[1],
                          iss_radius_src=0.3 + 0.1 * rng.random(), iss_radius_tgt=0.3 + 0.1 * rng.random()))
    return pairs, dim


def run_arms(ctx, arms, reps):
    """warm-up, identical outputs, alternated timed repetitions, one profiled call per arm"""
    outs = {a: f() for a, f in arms.items()}
    first = next(iter(outs.values()))
    for a, o in outs.items():
        assert _bytes(o) == _bytes(first), "arm %s differs from the first arm" % a
    times = {a: [] for a in arms}
    for _ in range(reps):
        for a, f in arms.items():
            t = time.perf_counter()
            f()
            times[a].append((time.perf_counter() - t) * 1e3)
    stats = {}
    for a, f in arms.items():
        ctx.set_profiling(True)
        ctx.reset_stats()
        f()
        stats[a] = ctx.stats()
        ctx.set_profiling(False)
    return first, times, stats


def _bytes(o):
    if isinstance(o, tuple) and len(o) == 2 and isinstance(o[0], np.ndarray):
        return o[0].tobytes() + np.float32(o[1]).tobytes()
    return b"".join(_bytes(x) for x in o)


def summary(name, times, stats, dim, rows, pairs=None):
    """pairs: (query, train) pairs the candidate kernel scores, when b200m_get_stats cannot count them (batch calls count
    every query row against the whole concatenated train side)"""
    out = {"workload": name, "ms": {}, "ms_all": {}, "arms": {}}
    for a, v in times.items():
        s = stats[a]
        out["ms"][a] = round(statistics.median(v), 3)
        out["ms_all"][a] = [round(x, 3) for x in v]
        d = {"candidate_ms": round(s["ms_candidates"], 3), "rerank_ms": round(s["ms_rerank"], 3),
             "fallback_ms": round(s["ms_fallback"], 3), "candidate_launches": s["candidate_launches"],
             "rows_flagged": s["rows_flagged"], "candidates_per_row": round(s["candidates"] / max(rows, 1), 2)}
        if s["ms_candidates"] > 0:
            d["pairs_scored"] = pairs or s["pairs_scored"]
            tf = 2.0 * dim * d["pairs_scored"] / (s["ms_candidates"] * 1e-3) / 1e12
            d["candidate_tflops"] = round(tf, 1)
            d["share_of_1388"] = round(tf / PEAK_TFLOPS, 3)
        out["arms"][a] = d
    if "default" in out["ms"] and "exact" in out["ms"]:
        out["exact_over_default"] = round(out["ms"]["exact"] / out["ms"]["default"], 3)
    print(json.dumps(out), file=sys.stderr)
    return out


def pair_workload(ctx, name, src, tgt, dim, k, reps, arms_wanted):
    ctx.upload(0, src, dim)
    ctx.upload(1, tgt, dim)
    arms = {}
    if "default" in arms_wanted:
        arms["default"] = lambda: ctx.match(k, M.MODE_MUTUAL)
    if "exact" in arms_wanted:
        arms["exact"] = lambda: ctx.match(k, M.MODE_MUTUAL, precision=M.PREC_F32_EXACT)
    recs, times, stats = run_arms(ctx, arms, reps)
    return recs, summary(name, times, stats, dim, len(src) + len(tgt))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    name, power = card()
    rows = []
    want = lambda w: a.only is None or a.only == w   # noqa: E731
    with M.Context(0) as ctx:
        if want("usc20k"):
            src, tgt, dim = usc_rows(20000, 20000, 11)
            _, r = pair_workload(ctx, "usc-1960 20k x 20k k=1 mutual", src, tgt, dim, 1, a.reps, ("default", "exact"))
            rows.append(r)
        if want("usc100k"):
            src, tgt, dim = usc_rows(100000, 100000, 12)
            recs, r = pair_workload(ctx, "usc-1960 100k x 100k k=2 mutual", src, tgt, dim, 2, a.reps, ("default",))
            idx, dist, cnt = ctx.knn(2, 0)
            sample = np.random.default_rng(0).choice(len(src), 256, replace=False)
            ei, ed, ec = orc.knn(np.ascontiguousarray(src[sample, :dim]), np.ascontiguousarray(tgt[:, :dim]), 2)
            assert np.array_equal(idx[sample], ei) and np.array_equal(dist[sample], ed) and np.array_equal(cnt[sample], ec)
            r["sampled_rows_equal_oracle"] = 256
            rows.append(r)
            del src, tgt
        for d in (700, 1024):
            if want("dim%d" % d):
                src, tgt, dim = usc_rows(50000, 50000, 13, dim=d)
                _, r = pair_workload(ctx, "dim %d 50k x 50k k=1 mutual" % d, src, tgt, dim, 1, a.reps, ("default", "exact"))
                rows.append(r)
        if want("cluster"):
            pairs, dim = wide_pairs(5000, [1.0, 0.8], 16)
            arms = {"default": lambda: ctx.match_wide_batch(2, M.MODE_CLUSTER, pairs, dim),
                    "exact": lambda: ctx.match_wide_batch(2, M.MODE_CLUSTER, pairs, dim, precision=M.PREC_F32_EXACT)}
            _, times, stats = run_arms(ctx, arms, a.reps)
            rows_all = sum(len(x) for pr in pairs for sc in (pr["src_scales"], pr["tgt_scales"]) for x, _ in sc)
            scored = sum(2 * len(s) * len(t) for pr in pairs for (s, _), (t, _) in zip(pr["src_scales"], pr["tgt_scales"]))
            rows.append(summary("ClusterMatcher usc-1960 5k 2 scales k=2, 16 pairs (match_wide_batch)", times, stats, dim, rows_all,
                                scored))
    line = json.dumps({"tool": "bench_long_descriptors", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
