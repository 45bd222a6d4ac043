"""The device-resident batch calls against today's route for sets that already live in HBM, on the same seeded inputs.
Prints one JSON line.

    python tools/bench_batch_device.py [--reps N] [--out FILE]

Arms (alternated in one run, after a warm-up of each; host clock around calls that end in a device synchronise):
    via_host     the sets are CUDA tensors: copy each to a pinned host buffer, synchronise, then the host form
                 (Context.match_batch / match_wide_batch) -- what a caller with HBM-resident sets has to do today
    host_pinned  the host form on the pinned buffers alone: the floor of via_host
    device       the device form (GpuBackend.match_batch / match_wide_batch) on the CUDA tensors, records left in HBM,
                 then torch.cuda.synchronize()
Workloads (every pair distinct, so nothing is served twice from L2 in one call):
    match_batch      FPFH-33 20k x 20k, k = 1, mutual, B in {16, 64}                  (DESIGN.md section 3.11)
    LeftToRight      FPFH-33 20k keypoints, 3 scales (20k, 16k, 12k rows), k = 2, B = 16  (section 3.12)
    ClusterMatcher   SHOT-352 (1444-byte rows) 5k keypoints, 2 scales (5k, 4k rows), k = 2, B = 64
The device arm's records and averages are asserted identical to the host form's.  b200m_get_stats gives the launches per
call of each arm; a torch.profiler pass per arm, in a run of its own, gives the host -> device and device -> host bytes
that the arm's call moves (the via_host arm's device -> host copies of the sets included).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from lidar_global_registration_b200 import matcher as M   # noqa: E402
from lidar_global_registration_b200 import synth           # noqa: E402

# (name, kind, mode, descriptor, keypoints, rows per scale as a fraction of the keypoints, k, batch sizes)
WORKLOADS = [("match_batch fpfh 20k mutual", "pairs", M.MODE_MUTUAL, "fpfh", 20000, None, 1, [16, 64]),
             ("lr fpfh 20k 3 scales", "wide", M.MODE_MUTUAL, "fpfh", 20000, [1.0, 0.8, 0.6], 2, [16]),
             ("cluster shot 5k 2 scales", "wide", M.MODE_CLUSTER, "shot", 5000, [1.0, 0.8], 2, [64])]


def make_pairs(kind, desc, n, fracs, count):
    """host (numpy) pairs: (src, tgt) tuples, or the dicts of Context.match_wide_batch"""
    pairs, dim = [], None
    for i in range(count):
        if kind == "pairs":
            src, tgt, dim = synth.make_pair(desc, n, n, seed=4000 + i, nan_frac=0.001)
            pairs.append((src, tgt))
            continue
        rng = np.random.default_rng(800 + i)
        xyz = []
        for _ in range(2):
            x = np.zeros((n, 4), np.float32)
            x[:, :3] = rng.random((n, 3)) * 40
            x[: n // 4, :3] = x[0, :3] + 0.2 * rng.standard_normal((n // 4, 3)).astype(np.float32)
            xyz.append(x)
        s_sc, t_sc = [], []
        for s, f in enumerate(fracs):
            m = int(n * f)
            src, tgt, dim = synth.make_pair(desc, m, m, seed=5000 + 10 * i + s, nan_frac=0.001)
            maps = [None if m == n else np.sort(rng.choice(n, m, replace=False)).astype(np.int32) for _ in range(2)]
            s_sc.append((src, maps[0]))
            t_sc.append((tgt, maps[1]))
        pairs.append(dict(src_scales=s_sc, tgt_scales=t_sc, src_kps_xyz=xyz[0], tgt_kps_xyz=xyz[1],
                          iss_radius_src=0.3 + 0.1 * rng.random(), iss_radius_tgt=0.3 + 0.1 * rng.random()))
    return pairs, dim


def _map(pr, f):
    """apply f to every array of a pair (None stays None)"""
    g = lambda a: None if a is None else f(a)   # noqa: E731
    if isinstance(pr, tuple):
        return tuple(g(a) for a in pr)
    out = dict(pr)
    out["src_scales"] = [(g(a), g(m)) for a, m in pr["src_scales"]]
    out["tgt_scales"] = [(g(a), g(m)) for a, m in pr["tgt_scales"]]
    out["src_kps_xyz"], out["tgt_kps_xyz"] = g(pr["src_kps_xyz"]), g(pr["tgt_kps_xyz"])
    return out


def _tensors(pr):
    if isinstance(pr, tuple):
        return list(pr)
    return [a for sc in (pr["src_scales"], pr["tgt_scales"]) for t in sc for a in t if a is not None] + \
        [pr["src_kps_xyz"], pr["tgt_kps_xyz"]]


def transfer_bytes(fn):
    """torch.profiler over one call: bytes of the host -> device and device -> host copies in the trace"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        ev = json.load(open(path)).get("traceEvents", [])
    out = {"h2d_bytes": 0, "d2h_bytes": 0, "h2d_copies": 0, "d2h_copies": 0}
    for e in ev:
        if e.get("cat") != "gpu_memcpy":
            continue
        b = int(e.get("args", {}).get("bytes", 0))
        if "HtoD" in e.get("name", ""):
            out["h2d_bytes"] += b
            out["h2d_copies"] += 1
        elif "DtoH" in e.get("name", ""):
            out["d2h_bytes"] += b
            out["d2h_copies"] += 1
    return out


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = r.stdout.strip().splitlines()[0].rsplit(",", 1)
    return name.strip(), power.strip()


def main():
    import torch
    from lidar_global_registration_b200 import device as D
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = card()
    rows = []
    b = D.GpuBackend(0)
    dev = b.device
    with M.Context(0) as ctx:
        for wname, kind, mode, desc, n, fracs, k, batches in WORKLOADS:
            host_all, dim = make_pairs(kind, desc, n, fracs, max(batches))
            dev_all = [_map(pr, lambda x: torch.from_numpy(x).to(dev)) for pr in host_all]
            pin_all = [_map(pr, lambda x: torch.from_numpy(x).pin_memory()) for pr in host_all]
            torch.cuda.synchronize()
            for B in batches:
                d_pairs, p_pairs = dev_all[:B], pin_all[:B]
                np_pairs = [_map(pr, lambda t: t.numpy()) for pr in p_pairs]
                copies = [(s, d) for pp, dp in zip(p_pairs, d_pairs) for s, d in zip(_tensors(pp), _tensors(dp))]
                set_bytes = sum(d.numel() * d.element_size() for _, d in copies)
                if kind == "pairs":
                    host = lambda: ctx.match_batch(k, mode, np_pairs, dim)             # noqa: E731
                    devf = lambda: b.match_batch(k, mode, d_pairs, dim)               # noqa: E731
                else:
                    host = lambda: ctx.match_wide_batch(k, mode, np_pairs, dim)        # noqa: E731
                    devf = lambda: b.match_wide_batch(k, mode, d_pairs, dim)          # noqa: E731

                def via_host():
                    for s, d in copies:
                        s.copy_(d, non_blocking=True)
                    torch.cuda.synchronize()
                    return host()

                def device():
                    r = devf()
                    torch.cuda.synchronize()
                    return r

                ref, _, got = via_host(), host(), device()                           # warm-up of every arm
                for (r0, a0), (r1, a1) in zip(ref, got):
                    assert r1.cpu().numpy().view(M.CORR_DTYPE).reshape(-1).tobytes() == r0.tobytes(), "device and host forms differ"
                    assert np.float32(a0).tobytes() == np.float32(a1).tobytes(), "device and host averages differ"
                arms = {"via_host": via_host, "host_pinned": host, "device": device}
                times = {k_: [] for k_ in arms}
                for _ in range(a.reps):
                    for arm, f in arms.items():
                        t = time.perf_counter()
                        f()
                        times[arm].append(time.perf_counter() - t)
                launches = {}
                for arm, f in arms.items():
                    c = b.ctx if arm == "device" else ctx
                    c.reset_stats()
                    f()
                    launches[arm] = c.stats()["launches"]
                xfer = {arm: transfer_bytes(f) for arm, f in arms.items()}
                med = {arm: statistics.median(v) * 1e3 for arm, v in times.items()}
                rows.append({
                    "workload": wname, "mode": mode, "k": k, "keypoints": n, "scales": len(fracs) if fracs else 1, "pairs": B,
                    "set_bytes": set_bytes, "records": sum(len(r) for r, _ in ref),
                    "ms": {arm: round(v, 3) for arm, v in med.items()},
                    "ms_all": {arm: [round(x * 1e3, 3) for x in v] for arm, v in times.items()},
                    "host_pinned_over_device": round(med["host_pinned"] / med["device"], 3),
                    "via_host_over_device": round(med["via_host"] / med["device"], 3),
                    "launches": launches, "transfers": xfer,
                })
                print("%-30s B=%-3d via_host %8.2f ms  host_pinned %8.2f ms  device %8.2f ms  launches %s  h2d %s" % (
                    wname, B, med["via_host"], med["host_pinned"], med["device"], launches,
                    {arm: x["h2d_bytes"] for arm, x in xfer.items()}), file=sys.stderr)
            del dev_all, pin_all
            torch.cuda.empty_cache()
    b.close()
    line = json.dumps({"tool": "bench_batch_device", "gpu": name, "power_limit": power, "reps": a.reps, "results": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
