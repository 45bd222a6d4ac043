"""Batch calls (b200m_knn_batch / b200m_match_batch): every pair's output must equal, byte for byte, upload + knn / match
on that pair alone (and the oracle on the small cases).  The GPU tests run with -m gpu on a B200; the layout of the C
struct and the C++ test program's build are checked without one."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from lidar_global_registration_b200 import build as b200_build
from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "batch_test")
gpu = pytest.mark.gpu

# pair sizes on both sides of every boundary of the layout: a 32-row chunk, a 256-row tile / CTA pair of query rows
SIZES = [0, 1, 31, 32, 255, 256, 257, 3000]
MODES = [M.MODE_ONE_SIDED, M.MODE_MUTUAL, M.MODE_RATIO, M.MODE_RATIO_MUTUAL]
ORACLE_MODE = {M.MODE_ONE_SIDED: "one_sided", M.MODE_MUTUAL: "mutual", M.MODE_RATIO: "ratio"}


def _pair(desc, ns, nt, seed):
    s, t, dim = synth.make_pair(desc, max(ns, 1), max(nt, 1), seed=seed, nan_frac=0.01)
    return np.ascontiguousarray(s[:ns]), np.ascontiguousarray(t[:nt]), dim


def _boundary_pairs(desc, extra=()):
    """every size of SIZES on both sides (an empty source and an empty target among them), a target with fewer valid rows
    than k, all-NaN sets on either side, then `extra` (ns, nt) pairs"""
    shapes = list(zip(SIZES, SIZES[3:] + SIZES[:3])) + [(40, 3), (50, 60), (70, 40)] + list(extra)
    pairs = []
    for i, (ns, nt) in enumerate(shapes):
        s, t, dim = _pair(desc, ns, nt, 100 + i)
        if (ns, nt) == (40, 3):
            t[0, 0] = np.nan        # two valid target rows
        if (ns, nt) == (50, 60):
            s[:, :] = np.nan
        if (ns, nt) == (70, 40):
            t[:, :] = np.nan
        pairs.append((s, t))
    return pairs, dim


def _modes(k):
    return [m for m in MODES if k >= 2 or m in (M.MODE_ONE_SIDED, M.MODE_MUTUAL)]


def _single(ctx, pairs, dim, k, modes, **kw):
    """per pair: upload both sets, knn (direction 0) and match in every mode -- what a loop over pairs computes"""
    out = []
    for s, t in pairs:
        ctx.upload(0, s, dim)
        ctx.upload(1, t, dim)
        out.append((ctx.knn(k, 0, **kw), {m: ctx.match(k, m, **kw) for m in modes}))
    return out


def _same_lists(a, b):
    assert len(a) == 3 and len(b) == 3
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()


def _check_batch(ctx, pairs, dim, k, modes, oracle=False, **kw):
    knn = ctx.knn_batch(k, pairs, dim, **kw)
    got = {m: ctx.match_batch(k, m, pairs, dim, **kw) for m in modes}
    ref = _single(ctx, pairs, dim, k, modes, **kw)
    assert len(knn) == len(pairs)
    for p, (s, t) in enumerate(pairs):
        _same_lists(knn[p], ref[p][0])
        idx, _, cnt = knn[p]
        assert idx.shape == (len(s), k)
        assert np.all((idx == -1) | ((idx >= 0) & (idx < len(t))))   # never a gap row, never another pair's row
        assert np.all(idx[np.arange(k)[None, :] >= cnt[:, None]] == -1)
        for m in modes:
            recs, avg = got[m][p]
            rrecs, ravg = ref[p][1][m]
            assert recs.tobytes() == rrecs.tobytes() and avg == ravg, (p, m)
            assert np.all((recs["index_query"] >= 0) & (recs["index_query"] < len(s)))
            assert np.all((recs["index_match"] >= 0) & (recs["index_match"] < len(t)))
        if oracle and len(s) and len(t):
            sd, td = s[:, :dim], t[:, :dim]
            _same_lists(knn[p], orc.knn(sd, td, k))
            for m in modes:
                if m in ORACLE_MODE:
                    e, eavg = orc.match(sd, td, k, ORACLE_MODE[m], distance_thr=np.float32(M.FLT_MAX))
                    assert got[m][p][0].tobytes() == e.tobytes() and got[m][p][1] == np.float32(eavg), (p, m)
    return knn, got


# ---- without a GPU ------------------------------------------------------------------------------------------------------
def test_pair_struct_is_the_c_layout():
    assert ctypes.sizeof(M._Pair) == 32


def _build_exe():
    b200_build.build()
    src = os.path.join(ROOT, "tests", "cpp", "batch_test.cpp")
    deps = [src, os.path.join(ROOT, "include", "b200match_shim.hpp"), os.path.join(ROOT, "include", "b200match.h")]
    if os.path.exists(EXE) and all(os.path.getmtime(EXE) >= os.path.getmtime(d) for d in deps):
        return EXE
    libdir = os.path.join(ROOT, "lidar_global_registration_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                    "-L", libdir, "-l:libb200match.so", "-Wl,-rpath," + libdir], check=True)
    return EXE


def test_batch_program_compiles_and_links():
    r = subprocess.run([_build_exe()], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


# ---- on the GPU -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [1, 2, 5])
@pytest.mark.parametrize("desc", ["fpfh", "shot", "rops"])
def test_batch_equals_single_pairs_and_oracle(desc, k):
    """FPFH runs the chunk-entry split-N candidate kernel, SHOT and RoPS the four-warp (EH = 1) kernels."""
    pairs, dim = _boundary_pairs(desc)
    with M.Context(0) as ctx:
        _check_batch(ctx, pairs, dim, k, _modes(k), oracle=True)


@gpu
def test_batch_thresholds_per_pair():
    pairs, dim = _boundary_pairs("fpfh")
    rng = np.random.default_rng(7)
    ts = [rng.random(len(s)).astype(np.float32) for s, _ in pairs]
    tt = [rng.random(len(t)).astype(np.float32) for _, t in pairs]
    with M.Context(0) as ctx:
        for mode in (M.MODE_ONE_SIDED, M.MODE_MUTUAL):
            got = ctx.match_batch(2, mode, pairs, dim, distance_thr=0.9, thr_src=ts, thr_tgt=tt)
            for p, (s, t) in enumerate(pairs):
                ctx.upload(0, s, dim)
                ctx.upload(1, t, dim)
                recs, avg = ctx.match(2, mode, distance_thr=0.9, thr_src=ts[p], thr_tgt=tt[p])
                assert got[p][0].tobytes() == recs.tobytes() and got[p][1] == avg


@gpu
def test_mixed_batch_large_and_small_pairs():
    """one 60k x 60k pair next to 40 small ones: the small pairs have far fewer train tiles than the launch has splits,
    so most of their CTAs have nothing to sweep"""
    rng = np.random.default_rng(11)
    s, t, dim = _pair("fpfh", 60000, 60000, 1)
    pairs = [(s, t)]
    for i in range(40):
        a, b, _ = _pair("fpfh", int(rng.integers(1, 3000)), int(rng.integers(1, 3000)), 200 + i)
        pairs.append((a, b))
    with M.Context(0) as ctx:
        _check_batch(ctx, pairs, dim, 1, [M.MODE_ONE_SIDED, M.MODE_MUTUAL])
        assert ctx.stats()["candidate_launches"] > 0


FORCED = [
    ({"B200M_TC_SPLITS": "3"}, {}, 2),            # 25-tile pair: three splits, one-tile pairs leave two CTAs empty
    ({"B200M_TC_SWEEP_LAG": "20"}, {}, 2),        # rotated sweep inside every segment
    ({"B200M_TC_ALT": "4"}, {}, 2),
    ({"B200M_TC_ALT": "5"}, {}, 5),
    ({}, {"cand_cap": "k"}, 5),                   # every overflowed row goes through the ranged exact kernels
    ({}, {"precision": M.PREC_F32_EXACT}, 2),     # the exact row kernel for every row
    ({}, {}, 20),                                 # k > 16: no tensor-core pass
]


@gpu
@pytest.mark.parametrize("env,kw,k", FORCED, ids=["splits3", "sweep_lag", "alt4", "alt5", "cap_k", "f32_exact", "k20"])
@pytest.mark.parametrize("desc", ["fpfh", "shot"])
def test_batch_forced_paths(monkeypatch, desc, env, kw, k):
    if desc == "shot" and any(e in env for e in ("B200M_TC_ALT", "B200M_TC_SWEEP_LAG")):
        pytest.skip("chunk-entry layouts and the rotated sweep belong to the one-atom (FPFH) kernel")
    for name, v in env.items():
        monkeypatch.setenv(name, v)
    kw = {n: (k if v == "k" else v) for n, v in kw.items()}
    pairs, dim = _boundary_pairs(desc, extra=[(300, 6200)])
    with M.Context(0) as ctx:
        _check_batch(ctx, pairs, dim, k, _modes(k)[:2], **kw)


@gpu
def test_single_pair_calls_after_a_batch():
    """the batch replaces the uploaded sets: a fresh upload + match afterwards is the single-pair answer (operand tensor
    maps, the prepared operands and the workspace sizes all follow the new sets)"""
    pairs, dim = _boundary_pairs("fpfh", extra=[(5000, 7000)])
    s, t, _ = _pair("fpfh", 1500, 2500, 42)
    with M.Context(0) as fresh:
        fresh.upload(0, s, dim)
        fresh.upload(1, t, dim)
        exp_knn = fresh.knn(2, 0)
        exp = fresh.match(2, M.MODE_MUTUAL)
    with M.Context(0) as ctx:
        ctx.match_batch(2, M.MODE_MUTUAL, pairs, dim)
        ctx.upload(0, s, dim)
        ctx.upload(1, t, dim)
        _same_lists(ctx.knn(2, 0), exp_knn)
        got = ctx.match(2, M.MODE_MUTUAL)
        assert got[0].tobytes() == exp[0].tobytes() and got[1] == exp[1]
        ctx.knn_batch(2, pairs, dim)
        ctx.upload(0, s, dim)
        ctx.upload(1, t, dim)
        _same_lists(ctx.knn(2, 0), exp_knn)


@gpu
def test_batch_errors(monkeypatch):
    pairs, dim = _boundary_pairs("fpfh")
    with M.Context(0) as ctx:
        with pytest.raises(M.B200MatchError, match="cluster"):
            ctx.match_batch(1, M.MODE_CLUSTER, pairs, dim)
        with pytest.raises(M.B200MatchError, match="b200m_knn_batch"):
            ctx.match_batch(1, M.MODE_KNN_ONLY, pairs, dim)
        L, p = ctx._L, M.Context._params(1, M.MODE_ONE_SIDED)
        keep, arr, stride, ns = M.Context._pairs(pairs, dim)
        offsets = np.zeros(len(pairs) + 1, np.uint64)
        out = np.empty(4, M.CORR_DTYPE)
        rc = L.b200m_match_batch(ctx._h, ctypes.byref(p), arr, len(pairs), stride, dim, None, None, out.ctypes.data, 4,
                                 offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), None)
        assert rc != 0 and "capacity too small" in L.b200m_last_error(ctx._h).decode()
        assert int(offsets[-1]) > 4 and np.all(np.diff(offsets.astype(np.int64)) >= 0)   # the sizes are reported
        arr[1].src = None    # a pair with source rows and no pointer
        rc = L.b200m_knn_batch(ctx._h, ctypes.byref(p), arr, len(pairs), stride, dim, None, None, None)
        assert rc != 0 and "null descriptor pointer in pair 1" in L.b200m_last_error(ctx._h).decode()
        assert ctx.knn_batch(1, [], dim) == [] and ctx.match_batch(1, M.MODE_MUTUAL, [], dim) == []
        empty = ctx.match_batch(1, M.MODE_MUTUAL, [(pairs[0][0], pairs[0][1])], dim)   # no source rows at all
        assert len(empty[0][0]) == 0 and empty[0][1] == M.FLT_MAX
    monkeypatch.setenv("B200M_TC_MODE", "mcast")
    monkeypatch.setenv("B200M_TC_CLUSTER", "4")
    with M.Context(0) as ctx:
        with pytest.raises(M.B200MatchError, match="B200M_TC_MODE=mcast"):
            ctx.match_batch(1, M.MODE_MUTUAL, pairs, dim)


@gpu
def test_cpp_batch_program_matches_oracle(tmp_path):
    exe = _build_exe()
    shapes = [(700, 900), (0, 50), (120, 0), (257, 31), (31, 257)]
    pairs = [_pair("fpfh", ns, nt, 300 + i)[:2] for i, (ns, nt) in enumerate(shapes)]
    sp, tp, op = tmp_path / "s.bin", tmp_path / "t.bin", tmp_path / "o.txt"
    np.concatenate([s for s, _ in pairs]).tofile(sp)
    np.concatenate([t for _, t in pairs]).tofile(tp)
    k = 2
    r = subprocess.run([exe, "fpfh", str(sp), str(tp), str(k), str(op)] + [str(n) for sh in shapes for n in sh],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    knn, match = {}, {}
    for line in open(op):
        w = line.split()
        if w[0] == "knn":
            knn[(int(w[1]), int(w[2]))] = [(int(a), np.float32(b)) for a, b in zip(w[4::2], w[5::2])]
        elif w[0] == "match":
            match.setdefault((w[1], int(w[2])), {"n": int(w[3]), "avg": np.float32(w[4]), "corr": []})
        elif w[0] == "corr":
            match[(w[1], int(w[2]))]["corr"].append((int(w[3]), int(w[4]), np.float32(w[5])))
    fmax = np.float32(np.finfo(np.float32).max)
    for p, (s, t) in enumerate(pairs):
        sd, td = s[:, :33], t[:, :33]
        if len(s) and len(t):
            idx, dist, cnt = orc.knn(sd, td, k)
            for i in range(len(s)):
                assert knn[(p, i)] == [(int(idx[i, m]), np.float32(dist[i, m])) for m in range(cnt[i])]
        else:
            assert all(knn[(p, i)] == [] for i in range(len(s)))
        for mode in ("one_sided", "mutual", "ratio"):
            got = match[(mode, p)]
            if len(s) and len(t):
                e, eavg = orc.match(sd, td, k, mode, distance_thr=np.float32(M.FLT_MAX))
                assert got["n"] == len(e) and got["avg"] == np.float32(eavg)
                assert got["corr"] == [(int(a), int(b), np.float32(c)) for a, b, c in
                                       zip(e["index_query"], e["index_match"], e["distance"])]
            else:
                assert got["n"] == 0 and got["avg"] == fmax
