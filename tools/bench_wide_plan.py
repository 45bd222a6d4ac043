"""Matcher-class batch plans against the device-resident batch call they bind, on the same seeded inputs already in HBM.
Prints one JSON line.

    python tools/bench_wide_plan.py [--reps N] [--out FILE]

Arms (alternated in one run after a warm-up of each; host clock around work that ends in a device synchronise):
    device   GpuBackend.match_wide_batch / match_wide_local_batch (b200m_match_multiscale(_local)_batch_device): per call
             the tables are built and uploaded, every tensor-core scale reads its prepare step back, and the result area is
             read back at the end
    plan     BatchPlan.run() then torch.cuda.synchronize(): the same work enqueued without the host
    graph    the plan's run captured once in a CUDA graph, replay() then torch.cuda.synchronize()
plus the host time to enqueue plan.run() and graph.replay() alone (no synchronise inside the timed window; the queue is
drained after it).  Each figure is the median of --reps alternated repetitions.
Workloads: what the reference's match_impl runs -- ClusterMatcher (its default) on SHOT-352 5k keypoints, 2 scales, k = 2,
B = 1 and 64; LeftToRightMatcher on FPFH-33 20k keypoints, 3 scales, k = 2, B = 16, without and with a guess (r = 4.7 over
keypoints in a 50 m box).  Every pair is distinct; scale 0 takes every keypoint (NULL maps), later scales a subset.
The plan's and the graph's records, offsets and averages are asserted identical to the device form's.
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

# (name, descriptor, keypoints per cloud, scales, k, mode, guess radius or None, batch sizes)
WORKLOADS = [("cluster shot 5k", "shot", 5000, 2, 2, M.MODE_CLUSTER, None, [1, 64]),
             ("mutual fpfh 20k", "fpfh", 20000, 3, 2, M.MODE_MUTUAL, None, [16]),
             ("mutual fpfh 20k guessed", "fpfh", 20000, 3, 2, M.MODE_MUTUAL, 4.7, [16])]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def same(got, ref, what):
    assert len(got) == len(ref)
    for p, ((r0, a0), (r1, a1)) in enumerate(zip(ref, got)):
        assert r1.cpu().numpy().tobytes() == r0.cpu().numpy().tobytes(), "%s: pair %d records differ" % (what, p)
        assert np.float32(a0).tobytes() == np.float32(a1).tobytes(), "%s: pair %d averages differ" % (what, p)


def wide_pair(torch, dev, desc, n, n_scales, seed):
    rng = np.random.default_rng(seed)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    xyz = []
    for _ in range(2):
        x = np.zeros((n, 4), np.float32)
        x[:, :3] = rng.random((n, 3)) * 50
        xyz.append(x)
    g = np.eye(4, dtype=np.float32)
    g[:3, 3] = rng.standard_normal(3)
    sides = ([], [])
    for s in range(n_scales):
        rows = n - 1000 * s * n // 20000
        src, tgt, dim = synth.make_pair(desc, rows, rows, seed=seed * 10 + s, nan_frac=0.001)
        for side, a in zip(sides, (src, tgt)):
            m = None if s == 0 else t(np.sort(rng.choice(n, rows, replace=False)).astype(np.int32))
            side.append((t(a), m))
    return dict(src_scales=sides[0], tgt_scales=sides[1], src_kps_xyz=t(xyz[0]), tgt_kps_xyz=t(xyz[1]),
                src_kps_moved=t(M.transform_keypoints(xyz[0], g)), tgt_kps_moved=t(M.transform_keypoints(xyz[1], M.invert_guess(g))),
                iss_radius_src=0.4, iss_radius_tgt=0.4), dim


def main():
    import torch
    from lidar_global_registration_b200 import device as D
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    b = D.GpuBackend(0)
    dev = b.device
    rows = []
    for wname, desc, n, n_scales, k, mode, radius, batches in WORKLOADS:
        pairs = []
        for i in range(max(batches)):
            pr, dim = wide_pair(torch, dev, desc, n, n_scales, 5000 + i)
            pairs.append(pr)
        torch.cuda.synchronize()
        for B in batches:
            d_pairs = pairs[:B]
            if radius is None:
                plan = b.plan_match_wide_batch(k, mode, d_pairs, dim)
                call = lambda: b.match_wide_batch(k, mode, d_pairs, dim)
            else:
                plan = b.plan_match_wide_local_batch(k, mode, d_pairs, radius, dim)
                call = lambda: b.match_wide_local_batch(k, mode, d_pairs, radius, dim)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                plan.run()

            def device():
                r = call()
                torch.cuda.synchronize()
                return r

            def run():
                plan.run()
                torch.cuda.synchronize()

            def replay():
                g.replay()
                torch.cuda.synchronize()

            ref = device()                                   # warm-up of every arm, and the outputs compared
            run()
            same(plan.results(), ref, "plan")
            plan.records.zero_()
            plan.offsets.zero_()
            replay()
            same(plan.results(), ref, "graph")
            arms = {"device": device, "plan": run, "graph": replay}
            enq = {"plan": plan.run, "graph": g.replay}
            times = {k_: [] for k_ in list(arms) + ["enqueue_plan", "enqueue_graph"]}
            for _ in range(a.reps):
                for arm, f in arms.items():
                    t = time.perf_counter()
                    f()
                    times[arm].append(time.perf_counter() - t)
                for arm, f in enq.items():
                    torch.cuda.synchronize()
                    t = time.perf_counter()
                    f()
                    times["enqueue_" + arm].append(time.perf_counter() - t)
                    torch.cuda.synchronize()
            same(plan.results(), ref, "after the timed repetitions")
            med = {arm: statistics.median(v) * 1e3 for arm, v in times.items()}
            rows.append({
                "workload": wname, "descriptor": desc, "keypoints": n, "scales": n_scales, "k": k,
                "mode": {M.MODE_CLUSTER: "cluster", M.MODE_MUTUAL: "mutual"}[mode], "guess_radius": radius, "pairs": B,
                "records": sum(len(r) for r, _ in ref),
                "ms": {arm: round(v, 4) for arm, v in med.items()},
                "ms_all": {arm: [round(x * 1e3, 4) for x in v] for arm, v in times.items()},
                "device_over_plan": round(med["device"] / med["plan"], 3),
                "device_over_graph": round(med["device"] / med["graph"], 3),
                "outputs_identical": True,
            })
            print("%-24s B=%-3d device %9.3f ms  plan %9.3f ms  graph %9.3f ms  enqueue plan %.3f ms  graph %.3f ms" % (
                wname, B, med["device"], med["plan"], med["graph"], med["enqueue_plan"], med["enqueue_graph"]),
                file=sys.stderr)
            del g
            plan.close()
        del pairs
        torch.cuda.empty_cache()
    b.close()
    line = json.dumps({"tool": "bench_wide_plan", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
