"""Batch plans with live counts on a stream of frames whose set sizes change, against the ways to answer such a stream
without them.  Prints one JSON line.

    python tools/bench_plan_rows.py [--reps N] [--frames F] [--out FILE]

Every pair's sets are bound once at capacity; a seeded stream of --frames frames draws every pair's live counts in
[cap/2, cap] (matcher classes: the live keypoints; scale 0, whose map is NULL, takes that many rows, a later scale the
prefix of its sorted map that points below them).  Arms, alternated in one run after a warm-up of each (host clock around
the whole stream, every frame ending in a device synchronise):
    device   the device form (GpuBackend.match_batch / match_wide_batch / match_wide_local_batch) on the live slices
    exact    a new exact-size plan per frame on the live slices (creation runs the batch once, synchronised, which answers
             the frame), then closed
    rows     one plan with live counts (rows= / kps_rows= and scale_rows=): the frame's counts copied device-to-device into
             the bound count tensors, run(), synchronise
    graph    the rows plan's run captured once in a CUDA graph: the same count copy, replay(), synchronise
Capacity overhead (same alternation, --runs runs per repetition): the rows plan at live = cap against an exact-size plan's
run() at cap, and at live = cap/2 against an exact-size plan's run() at cap/2.  Each figure is the median of --reps
repetitions.  Outputs (records, offsets, averages) of every frame are asserted identical across the four arms before timing.
Workloads (those of DESIGN.md sections 3.16-3.17): the match batch on FPFH-33 20k, mutual, k = 1, B = 1 and 16;
ClusterMatcher on SHOT-352 5k keypoints, 2 scales, k = 2, B = 16; LeftToRightMatcher guessed (r = 4.7) on FPFH-33 20k
keypoints, 3 scales, k = 2, B = 16 (the clouds of tools/bench_wide_plan.py).
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from lidar_global_registration_b200 import matcher as M   # noqa: E402
from lidar_global_registration_b200 import synth           # noqa: E402

# (name, kind, descriptor, keypoints / rows per set at capacity, scales, k, mode, guess radius, batch sizes)
WORKLOADS = [("match fpfh 20k mutual", "match", "fpfh", 20000, 0, 1, M.MODE_MUTUAL, None, [1, 16]),
             ("cluster shot 5k, 2 scales", "wide", "shot", 5000, 2, 2, M.MODE_CLUSTER, None, [16]),
             ("left-to-right fpfh 20k, 3 scales, guessed", "wide", "fpfh", 20000, 3, 2, M.MODE_MUTUAL, 4.7, [16])]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def same(got, ref, what):
    assert len(got) == len(ref)
    for p, ((r0, a0), (r1, a1)) in enumerate(zip(ref, got)):
        assert r1.cpu().numpy().tobytes() == r0.cpu().numpy().tobytes(), "%s: pair %d records differ" % (what, p)
        assert np.float32(a0).tobytes() == np.float32(a1).tobytes(), "%s: pair %d averages differ" % (what, p)


class MatchWork:
    """the match batch: a frame is one (source rows, target rows) per pair"""

    def __init__(self, b, torch, pairs, dim, k, mode):
        self.b, self.torch, self.pairs, self.dim, self.k, self.mode = b, torch, pairs, dim, k, mode
        self.live = torch.tensor([(p[0].shape[0], p[1].shape[0]) for p in pairs], dtype=torch.int32, device=b.device)

    def frame(self, rng, lo):
        return [(int(rng.integers(int(p[0].shape[0] * lo), p[0].shape[0] + 1)),
                 int(rng.integers(int(p[1].shape[0] * lo), p[1].shape[0] + 1))) for p in self.pairs]

    def scaled(self, f):
        return [(int(p[0].shape[0] * f), int(p[1].shape[0] * f)) for p in self.pairs]

    def device_counts(self, fr):
        return [self.torch.tensor(fr, dtype=self.torch.int32, device=self.b.device)]

    def sliced(self, fr):
        return [(s[:ns], t[:nt]) for (s, t), (ns, nt) in zip(self.pairs, fr)]

    def device(self, fr):
        return self.b.match_batch(self.k, self.mode, self.sliced(fr), self.dim)

    def exact_plan(self, fr):
        return self.b.plan_match_batch(self.k, self.mode, self.sliced(fr), self.dim)

    def rows_plan(self):
        return self.b.plan_match_batch(self.k, self.mode, self.pairs, self.dim, rows=self.live)

    def set_live(self, counts):
        self.live.copy_(counts[0])


class WideWork:
    """a matcher-class batch: a frame draws the live keypoints of every pair; scale 0 (a NULL map) takes that many rows,
    a later scale the prefix of its sorted map that points below the live keypoints"""

    def __init__(self, b, torch, pairs, dim, k, mode, radius):
        self.b, self.torch, self.pairs, self.dim, self.k, self.mode, self.radius = b, torch, pairs, dim, k, mode, radius
        self.maps = [[[None if m is None else m.cpu().numpy() for _, m in p[side]] for side in ("src_scales", "tgt_scales")]
                     for p in pairs]
        self.kps = torch.tensor([(p["src_kps_xyz"].shape[0], p["tgt_kps_xyz"].shape[0]) for p in pairs], dtype=torch.int32,
                                device=b.device)
        self.rows = torch.tensor([(p["src_scales"][s][0].shape[0], p["tgt_scales"][s][0].shape[0]) for p in pairs
                                  for s in range(len(p["src_scales"]))], dtype=torch.int32, device=b.device)

    def _rows(self, i, nk):
        return [tuple(int(nk[j]) if m is None else int(np.searchsorted(m, nk[j])) for j, m in enumerate(ms))
                for ms in zip(*self.maps[i])]

    def frame(self, rng, lo):
        out = []
        for i, p in enumerate(self.pairs):
            nk = [int(rng.integers(int(p[key].shape[0] * lo), p[key].shape[0] + 1)) for key in ("src_kps_xyz", "tgt_kps_xyz")]
            out.append((nk, self._rows(i, nk)))
        return out

    def scaled(self, f):
        out = []
        for i, p in enumerate(self.pairs):
            nk = [int(p[key].shape[0] * f) for key in ("src_kps_xyz", "tgt_kps_xyz")]
            out.append((nk, self._rows(i, nk)))
        return out

    def device_counts(self, fr):
        T, dev = self.torch, self.b.device
        return [T.tensor([nk for nk, _ in fr], dtype=T.int32, device=dev),
                T.tensor([r for _, rows in fr for r in rows], dtype=T.int32, device=dev)]

    def sliced(self, fr):
        out = []
        for p, (nk, rows) in zip(self.pairs, fr):
            d = dict(p)
            for j, side in enumerate(("src_scales", "tgt_scales")):
                d[side] = [(f_[:r[j]], None if m is None else m[:r[j]]) for (f_, m), r in zip(p[side], rows)]
            for key, n in (("src_kps_xyz", nk[0]), ("src_kps_moved", nk[0]), ("tgt_kps_xyz", nk[1]), ("tgt_kps_moved", nk[1])):
                d[key] = p[key][:n]
            out.append(d)
        return out

    def _call(self, pairs, plan, **kw):
        b = self.b
        if self.radius is None:
            return (b.plan_match_wide_batch if plan else b.match_wide_batch)(self.k, self.mode, pairs, self.dim, **kw)
        return (b.plan_match_wide_local_batch if plan else b.match_wide_local_batch)(self.k, self.mode, pairs, self.radius,
                                                                                      self.dim, **kw)

    def device(self, fr):
        return self._call(self.sliced(fr), False)

    def exact_plan(self, fr):
        return self._call(self.sliced(fr), True)

    def rows_plan(self):
        return self._call(self.pairs, True, kps_rows=self.kps, scale_rows=self.rows)

    def set_live(self, counts):
        self.kps.copy_(counts[0])
        self.rows.copy_(counts[1])


def main():
    import torch
    from lidar_global_registration_b200 import device as D
    import bench_wide_plan as BW
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    b = D.GpuBackend(0)
    dev = b.device
    rows_out = []
    for wname, kind, desc, n, n_scales, k, mode, radius, batches in WORKLOADS:
        pairs = []
        for i in range(max(batches)):
            if kind == "match":
                src, tgt, dim = synth.make_pair(desc, n, n, seed=5000 + i, nan_frac=0.001)
                pairs.append((torch.from_numpy(src).to(dev), torch.from_numpy(tgt).to(dev)))
            else:
                pr, dim = BW.wide_pair(torch, dev, desc, n, n_scales, 5000 + i)
                pairs.append(pr)
        torch.cuda.synchronize()
        for B in batches:
            w = MatchWork(b, torch, pairs[:B], dim, k, mode) if kind == "match" else WideWork(b, torch, pairs[:B], dim, k, mode,
                                                                                                 radius)
            rng = np.random.default_rng(B + n_scales)
            frames = [w.frame(rng, 0.5) for _ in range(a.frames)]
            d_frames = [w.device_counts(f) for f in frames]
            plan = w.rows_plan()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                plan.run()

            def device_frame(i):
                r = w.device(frames[i])
                torch.cuda.synchronize()
                return r

            def exact_frame(i):
                p = w.exact_plan(frames[i])
                torch.cuda.synchronize()
                return p

            def rows_frame(i):
                w.set_live(d_frames[i])
                plan.run()
                torch.cuda.synchronize()

            def graph_frame(i):
                w.set_live(d_frames[i])
                g.replay()
                torch.cuda.synchronize()

            for i in range(a.frames):   # warm-up of every arm, and the outputs compared frame by frame
                ref = device_frame(i)
                p = exact_frame(i)
                same(p.results(), ref, "exact frame %d" % i)
                p.close()
                rows_frame(i)
                same(plan.results(), ref, "rows frame %d" % i)
                plan.records.zero_()
                plan.offsets.zero_()
                graph_frame(i)
                same(plan.results(), ref, "graph frame %d" % i)

            def stream(f):
                def go():
                    for i in range(a.frames):
                        r = f(i)
                        if isinstance(r, D.BatchPlan):
                            r.close()
                return go

            arms = {"device": stream(device_frame), "exact": stream(exact_frame), "rows": stream(rows_frame),
                    "graph": stream(graph_frame)}
            # capacity overhead: exact-size plans at cap and cap/2 against the rows plan at those live counts
            full, half = w.scaled(1.0), w.scaled(0.5)
            ex_full, ex_half = w.exact_plan(full), w.exact_plan(half)
            d_full, d_half = w.device_counts(full), w.device_counts(half)
            for f, ex in ((d_full, ex_full), (d_half, ex_half)):   # same answers at both sizes
                w.set_live(f)
                plan.run()
                same(plan.results(), ex.results(), "capacity overhead")

            def runs(ex, f=None):
                def go():
                    if f is not None:
                        w.set_live(f)
                    for _ in range(a.runs):
                        (plan if f is not None else ex).run()
                    torch.cuda.synchronize()
                return go

            arms.update({"exact_cap": runs(ex_full), "rows_cap": runs(None, d_full), "exact_half": runs(ex_half),
                         "rows_half": runs(None, d_half)})
            for f in arms.values():
                f()
            times = {k_: [] for k_ in arms}
            for _ in range(a.reps):
                for arm, f in arms.items():
                    torch.cuda.synchronize()
                    t = time.perf_counter()
                    f()
                    times[arm].append(time.perf_counter() - t)
            per_frame = {arm: statistics.median(times[arm]) * 1e3 / a.frames for arm in ("device", "exact", "rows", "graph")}
            per_run = {arm: statistics.median(times[arm]) * 1e3 / a.runs for arm in ("exact_cap", "rows_cap", "exact_half",
                                                                                     "rows_half")}
            rows_out.append({
                "workload": wname, "descriptor": desc, "capacity": n, "scales": n_scales, "k": k, "mode": int(mode),
                "guess_radius": radius, "pairs": B, "frames": a.frames, "counts": "drawn in [cap/2, cap]",
                "ms_per_frame": {k_: round(v, 4) for k_, v in per_frame.items()},
                "ms_per_run": {k_: round(v, 4) for k_, v in per_run.items()},
                "ms_all": {k_: [round(x * 1e3, 4) for x in v] for k_, v in times.items()},
                "device_over_rows": round(per_frame["device"] / per_frame["rows"], 3),
                "device_over_graph": round(per_frame["device"] / per_frame["graph"], 3),
                "exact_over_rows": round(per_frame["exact"] / per_frame["rows"], 3),
                "overhead_at_cap": round(per_run["rows_cap"] / per_run["exact_cap"], 3),
                "overhead_at_half": round(per_run["rows_half"] / per_run["exact_half"], 3),
                "outputs_identical": True,
            })
            print("%-42s B=%-3d per frame: device %8.3f  exact %8.3f  rows %8.3f  graph %8.3f ms | per run: cap exact %.3f "
                  "rows %.3f, cap/2 exact %.3f rows %.3f ms" % (wname, B, per_frame["device"], per_frame["exact"],
                                                                per_frame["rows"], per_frame["graph"], per_run["exact_cap"],
                                                                per_run["rows_cap"], per_run["exact_half"], per_run["rows_half"]),
                  file=sys.stderr)
            del g
            plan.close()
            ex_full.close()
            ex_half.close()
        del pairs
        torch.cuda.empty_cache()
    b.close()
    line = json.dumps({"tool": "bench_plan_rows", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows_out})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
