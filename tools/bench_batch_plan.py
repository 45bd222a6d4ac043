"""Batch plans against the device-resident batch call they bind, on the same seeded inputs already in HBM.  Prints one JSON
line.

    python tools/bench_batch_plan.py [--reps N] [--out FILE]

Arms (alternated in one run after a warm-up of each; host clock around work that ends in a device synchronise):
    device   GpuBackend.match_batch (b200m_match_batch_device): two host round trips per call, tables built per call
    plan     BatchPlan.run() then torch.cuda.synchronize(): the same work enqueued without the host
    graph    the plan's run captured once in a CUDA graph, replay() then torch.cuda.synchronize()
plus the host time to enqueue plan.run() and graph.replay() alone (no synchronise inside the timed window; the queue is
drained after it).  Each figure is the median of --reps alternated repetitions.
Workloads: FPFH-33 20k x 20k, k = 1, mutual, B in {1, 16, 64} (§3.11: a single pair is about one wave of the candidate
kernel, so fixed cost per call shows); SHOT-352 (1444-byte rows) 5k x 5k, k = 2, mutual, B = 64.  Every pair is distinct.
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

# (name, descriptor, rows per set, k, batch sizes)
WORKLOADS = [("fpfh 20k mutual", "fpfh", 20000, 1, [1, 16, 64]), ("shot 5k mutual", "shot", 5000, 2, [64])]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def same(got, ref, what):
    assert len(got) == len(ref)
    for p, ((r0, a0), (r1, a1)) in enumerate(zip(ref, got)):
        assert r1.cpu().numpy().tobytes() == r0.cpu().numpy().tobytes(), "%s: pair %d records differ" % (what, p)
        assert np.float32(a0).tobytes() == np.float32(a1).tobytes(), "%s: pair %d averages differ" % (what, p)


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
    for wname, desc, n, k, batches in WORKLOADS:
        pairs = []
        for i in range(max(batches)):
            src, tgt, dim = synth.make_pair(desc, n, n, seed=4000 + i, nan_frac=0.001)
            pairs.append((torch.from_numpy(src).to(dev), torch.from_numpy(tgt).to(dev)))
        torch.cuda.synchronize()
        for B in batches:
            d_pairs = pairs[:B]
            plan = b.plan_match_batch(k, M.MODE_MUTUAL, d_pairs, dim)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                plan.run()

            def device():
                r = b.match_batch(k, M.MODE_MUTUAL, d_pairs, dim)
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
            med = {arm: statistics.median(v) * 1e3 for arm, v in times.items()}
            rows.append({
                "workload": wname, "descriptor": desc, "rows": n, "k": k, "mode": "mutual", "pairs": B,
                "records": sum(len(r) for r, _ in ref),
                "ms": {arm: round(v, 4) for arm, v in med.items()},
                "ms_all": {arm: [round(x * 1e3, 4) for x in v] for arm, v in times.items()},
                "device_over_plan": round(med["device"] / med["plan"], 3),
                "device_over_graph": round(med["device"] / med["graph"], 3),
                "outputs_identical": True,
            })
            print("%-18s B=%-3d device %8.3f ms  plan %8.3f ms  graph %8.3f ms  enqueue plan %.3f ms  graph %.3f ms" % (
                wname, B, med["device"], med["plan"], med["graph"], med["enqueue_plan"], med["enqueue_graph"]),
                file=sys.stderr)
            del g
            plan.close()
        del pairs
        torch.cuda.empty_cache()
    b.close()
    line = json.dumps({"tool": "bench_batch_plan", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
