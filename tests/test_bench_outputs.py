"""bench.py --dump-outputs: the arrays the timed step returned, as .npy files a later build can be compared against."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from lidar_global_registration_b200 import matcher as M  # noqa: E402


def _records(n_rows, per_row, seed):
    rng = np.random.default_rng(seed)
    q = np.repeat(np.arange(n_rows), rng.integers(0, per_row + 1, n_rows))     # ascending, at most per_row per row
    rec = np.zeros(q.shape[0], M.CORR_DTYPE)
    rec["index_query"], rec["index_match"] = q, rng.integers(0, 10 ** 6, q.shape[0])
    rec["distance"], rec["threshold"] = rng.random(q.shape[0]), np.float32(M.FLT_MAX)
    return rec


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_records_are_written_whole_when_they_fit(tmp_path):
    rec = _records(1000, 2, 1)
    assert bench.write_outputs(str(tmp_path), 1000, records=rec, per_row=2) == ["distance", "index_match", "index_query", "threshold"]
    got = _load(tmp_path)
    for name in ("index_query", "index_match"):
        assert got[name].dtype == np.float64 and np.array_equal(got[name], rec[name])
    for name in ("distance", "threshold"):
        assert got[name].dtype == np.float32 and np.array_equal(got[name], rec[name])


def test_large_outputs_are_a_seeded_row_sample_under_the_size_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 200000)
    n, k = 20000, 3
    sizes, rows = [], []
    for i, rec in enumerate((_records(n, k, 2), _records(n, k, 3))):   # two different results: the same rows
        d = tmp_path / str(i)
        bench.write_outputs(str(d), n, records=rec, per_row=k)
        got = _load(d)
        r = got["query_rows"].astype(np.int64)
        assert 0 < r.shape[0] < n and np.all(np.diff(r) > 0)
        keep = np.isin(rec["index_query"], r)
        assert np.array_equal(got["index_query"], rec["index_query"][keep]) and np.array_equal(got["distance"], rec["distance"][keep])
        sizes.append(sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)))
        rows.append(r)
    assert np.array_equal(rows[0], rows[1])
    assert max(sizes) <= 200000 + 5 * 128                                  # + the .npy headers
    lists = (np.zeros((n, k), np.int32), np.ones((n, k), np.float32), np.full(n, k, np.int32))
    bench.write_outputs(str(tmp_path / "lists"), n, lists=lists)
    got = _load(tmp_path / "lists")
    assert got["knn_index"].dtype == np.float64 and got["knn_distance"].dtype == np.float32
    assert got["knn_index"].shape == (got["query_rows"].shape[0], k) and np.all(got["knn_count"] == k)


def test_dump_needs_the_gpu_arm():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_dumped_outputs_are_the_oracle_correspondences(tmp_path):
    """C1 (FPFH-33 20k x 20k, k=1, mutual) through bench.py: the dumped records are the oracle's for the same seeded inputs,
    and as many as the JSON line reports."""
    import torch
    from lidar_global_registration_b200 import synth
    from oracle import oracle as orc
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout)
    desc, n_src, n_tgt, k, mode, _ = bench.WORKLOADS["c1"]
    src, tgt, dim = synth.make_pair_torch(desc, n_src, n_tgt, torch.device("cuda", 0))
    src, tgt = src.cpu().numpy(), tgt.cpu().numpy()
    exp, _ = orc.match(src[:, :dim], tgt[:, :dim], k, mode, distance_thr=np.float32(M.FLT_MAX))
    got = _load(tmp_path)
    assert sorted(got) == ["distance", "index_match", "index_query", "threshold"]
    assert got["index_query"].shape[0] == line["correspondences"] == len(exp) > 0
    for name in exp.dtype.names:
        assert np.array_equal(got[name], exp[name]), name
