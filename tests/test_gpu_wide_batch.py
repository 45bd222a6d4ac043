"""b200m_match_multiscale_batch (Context.match_wide_batch, match_many, b200match::matchMany): every pair's records and
average must equal, byte for byte, b200m_match_multiscale on that pair alone (Context.match_wide), and the oracle on the
small cases.  The GPU tests run with -m gpu on a B200; the C struct layout and the C++ program's build are checked
without one."""
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
EXE = os.path.join(ROOT, "tests", "cpp", "wide_batch_test")
gpu = pytest.mark.gpu

GMODE = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "cluster": M.MODE_CLUSTER}
MATCHING_ID = {"one_sided": M.MATCHING_ONE_SIDED, "mutual": M.MATCHING_LEFT_TO_RIGHT, "cluster": M.MATCHING_CLUSTER}
DTHR = np.float32(0.7)


def _xyz(rng, n):
    """keypoints (pcl::PointXYZ rows, 16 B) with a tight cluster, so that the vote and the cluster filter matter"""
    x = np.zeros((n, 4), np.float32)
    x[:, :3] = rng.random((n, 3)) * 4
    if n:
        x[: n // 4, :3] = x[0, :3] + 0.02 * rng.standard_normal((n // 4, 3)).astype(np.float32)
    return x


def _case(desc, k, n_scales, seed, n_sk=800, n_tk=950, rows=None, identity=None, sx=None, tx=None):
    """one cloud pair as match_wide takes it: per scale a subset of the keypoints (index maps) or all of them (None).
    rows: optional [(source rows, target rows)] per scale (maps are then random subsets of that size, or identity)."""
    rng = np.random.default_rng(seed)
    sx = _xyz(rng, n_sk) if sx is None else sx
    tx = _xyz(rng, n_tk) if tx is None else tx
    s_sc, t_sc, dim = [], [], None
    for s in range(n_scales):
        ns, nt = rows[s] if rows else (n_sk - 50 * s, n_tk - 40 * s)
        ident = identity if identity is not None else (n_scales == 1 and k == 1)
        smap = None if ident and ns == n_sk else np.sort(rng.choice(n_sk, ns, replace=False)).astype(np.int32)
        tmap = None if ident and nt == n_tk else np.sort(rng.choice(n_tk, nt, replace=False)).astype(np.int32)
        src, tgt, dim = synth.make_pair(desc, max(ns, 1), max(nt, 1), seed=1000 * seed + s, nan_frac=0.01)
        s_sc.append((np.ascontiguousarray(src[:ns, :dim]), smap))
        t_sc.append((np.ascontiguousarray(tgt[:nt, :dim]), tmap))
    if dim is None:
        dim = synth.DESCRIPTORS[desc][0]
    pr = dict(src_scales=s_sc, tgt_scales=t_sc, src_kps_xyz=sx, tgt_kps_xyz=tx,
              iss_radius_src=np.float32(0.03 + 0.05 * rng.random()), iss_radius_tgt=np.float32(0.03 + 0.05 * rng.random()))
    return pr, rng.random(n_sk).astype(np.float32), rng.random(n_tk).astype(np.float32), dim


def _single(ctx, k, mode, pr, dim, ts, tt, **kw):
    if not pr["src_scales"]:   # no scale: no candidates at all
        return np.empty(0, M.CORR_DTYPE), M.FLT_MAX
    return ctx.match_wide(k, mode, pr["src_scales"], pr["tgt_scales"], pr["src_kps_xyz"], pr["tgt_kps_xyz"], pr["iss_radius_src"],
                          pr["iss_radius_tgt"], dim, 40, DTHR, ts, tt, **kw)


def _oracle(mode, k, pr, ts, tt):
    return orc.match_wide(mode, pr["src_scales"], pr["tgt_scales"], pr["src_kps_xyz"][:, :3], pr["tgt_kps_xyz"][:, :3],
                          pr["iss_radius_src"], pr["iss_radius_tgt"], k, 40, DTHR, ts, tt)


def _check(mode, k, cases, oracle=False, single_env=None, monkeypatch=None, **kw):
    pairs = [c[0] for c in cases]
    ts, tt = [c[1] for c in cases], [c[2] for c in cases]
    dim = cases[0][3]
    with M.Context(0) as ctx:
        got = ctx.match_wide_batch(k, GMODE[mode], pairs, dim, 40, DTHR, ts, tt, **kw)
    for name, v in (single_env or {}).items():
        monkeypatch.setenv(name, v)
    with M.Context(0) as ctx:
        ref = [_single(ctx, k, GMODE[mode], pr, dim, a, b, **kw) for pr, a, b in zip(pairs, ts, tt)]
    assert len(got) == len(pairs)
    for p, ((recs, avg), (rrecs, ravg)) in enumerate(zip(got, ref)):
        assert recs.tobytes() == rrecs.tobytes() and avg == ravg, (mode, p)
        n_s, n_t = len(pairs[p]["src_kps_xyz"]), len(pairs[p]["tgt_kps_xyz"])
        assert np.all((recs["index_query"] >= 0) & (recs["index_query"] < n_s))
        assert np.all((recs["index_match"] >= 0) & (recs["index_match"] < n_t))
        if oracle and n_s and n_t and pairs[p]["src_scales"]:
            e, eavg = _oracle(mode, k, pairs[p], ts[p], tt[p])
            assert recs.tobytes() == e.tobytes() and avg == eavg, (mode, p)
    return got


# ---- without a GPU ------------------------------------------------------------------------------------------------------
def test_wide_pair_struct_is_the_c_layout(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "b200match.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(b200m_wide_pair));\n' +
                   "".join('  printf(" %%zu", offsetof(b200m_wide_pair, %s));\n' % n for n, _ in M._WidePair._fields_) +
                   '  printf(" %zu\\n", sizeof(b200m_scale));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[0] == ctypes.sizeof(M._WidePair)
    assert got[1:-1] == [getattr(M._WidePair, n).offset for n, _ in M._WidePair._fields_]
    assert got[-1] == ctypes.sizeof(M._Scale)


def _build_exe():
    b200_build.build()
    src = os.path.join(ROOT, "tests", "cpp", "wide_batch_test.cpp")
    deps = [src, os.path.join(ROOT, "include", "b200match_shim.hpp"), os.path.join(ROOT, "include", "b200match.h")]
    if os.path.exists(EXE) and all(os.path.getmtime(EXE) >= os.path.getmtime(d) for d in deps):
        return EXE
    libdir = os.path.join(ROOT, "lidar_global_registration_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                    "-L", libdir, "-l:libb200match.so", "-Wl,-rpath," + libdir], check=True)
    return EXE


def test_wide_batch_program_compiles_and_links():
    r = subprocess.run([_build_exe()], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


# ---- on the GPU -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
@pytest.mark.parametrize("desc,k,n_scales", [("fpfh", 1, 1), ("fpfh", 2, 1), ("shot", 2, 2), ("rops", 3, 3), ("fpfh", 5, 2)])
def test_wide_batch_equals_single_pairs_and_oracle(desc, k, n_scales, mode):
    cases = [_case(desc, k, n_scales, 31 + 7 * k + n_scales),
             _case(desc, k, n_scales, 5, n_sk=300, n_tk=420),
             _case(desc, k, n_scales, 6, n_sk=600, n_tk=257, identity=False)]
    got = _check(mode, k, cases, oracle=True)
    assert sum(len(r) for r, _ in got) > 0


def _edge_cases(k):
    d = "fpfh"
    return [
        _case(d, k, 2, 40),                                                    # an ordinary pair
        _case(d, k, 1, 41, n_sk=300, n_tk=256, identity=True),                  # NULL maps
        _case(d, k, 3, 42, n_sk=400, n_tk=380, rows=[(400, 380), (0, 0), (350, 300)]),   # an empty scale in the middle
        _case(d, k, 1, 43, n_sk=0, n_tk=100, rows=[(0, 100)]),                  # no source keypoints
        _case(d, k, 1, 44, n_sk=200, n_tk=0, rows=[(200, 0)]),                  # no target keypoints
        _case(d, k, 1, 45, n_sk=20, n_tk=30, identity=True),                    # fewer keypoints than cluster_k
        _case(d, k, 2, 46, n_sk=257, n_tk=256, rows=[(255, 256), (257, 255)], identity=True),   # 255 / 256 / 257 rows
        _case(d, k, 2, 47, n_sk=500, n_tk=520),                                # all-NaN scale (below)
        _case(d, k, 0, 48, n_sk=50, n_tk=60),                                   # no scale at all
        _case(d, k, 3, 49, n_sk=700, n_tk=650),                                 # more scales than most
    ]


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
def test_wide_batch_edge_case_pairs(mode):
    cases = _edge_cases(2)
    cases[7][0]["src_scales"][1][0][:, :] = np.nan
    got = _check(mode, 2, cases, oracle=True)
    assert len(got[3][0]) == 0 and got[3][1] == M.FLT_MAX      # no source keypoints
    assert len(got[4][0]) == 0                                 # no target keypoints
    assert len(got[8][0]) == 0 and got[8][1] == M.FLT_MAX      # no scale
    assert len(got[0][0]) > 0 and len(got[9][0]) > 0


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
def test_wide_batch_pairs_stay_isolated(mode):
    """every pair has the SAME keypoint coordinates: a 3-D neighbourhood or a vote that crossed pairs would pick another
    pair's keypoints (ties go to the lower, earlier pair's id); then two pairs swap their radii"""
    rng = np.random.default_rng(3)
    sx, tx = _xyz(rng, 600), _xyz(rng, 640)
    cases = [_case("fpfh", 2, 2, 60 + i, n_sk=600, n_tk=640, sx=sx, tx=tx) for i in range(4)]
    _check(mode, 2, cases)
    a, b = cases[0][0], cases[1][0]
    a["iss_radius_src"], b["iss_radius_src"] = b["iss_radius_src"], a["iss_radius_src"]
    a["iss_radius_tgt"], b["iss_radius_tgt"] = b["iss_radius_tgt"], a["iss_radius_tgt"]
    _check(mode, 2, cases)


FORCED = [({"B200M_TC_SPLITS": "3"}, {}, {}), ({}, {"precision": M.PREC_F32_EXACT}, {}), ({}, {}, {"B200M_MASKED_MIN_PAIRS": "1"})]


@gpu
@pytest.mark.parametrize("env,kw,single_env", FORCED, ids=["splits3", "f32_exact", "masked_single"])
def test_wide_batch_forced_paths(monkeypatch, env, kw, single_env):
    for name, v in env.items():
        monkeypatch.setenv(name, v)
    cases = [_case("fpfh", 1, 1, 70 + i, n_sk=300 + 200 * i, n_tk=900 - 150 * i) for i in range(4)]
    if single_env:   # the masked reverse pass of a single-scale mutual call gives the same output
        _check("mutual", 1, cases, single_env=single_env, monkeypatch=monkeypatch)
        return
    for mode in ("one_sided", "mutual", "cluster"):
        _check(mode, 1, cases, **kw)
        _check(mode, 2, [_case("fpfh", 2, 2, 90 + i, n_sk=500, n_tk=450) for i in range(3)], **kw)


class _CapOne:
    """the library with cap = 1 in b200m_match_multiscale_batch, recording the offsets it fills"""

    def __init__(self, L, n_pairs):
        self.L, self.n_pairs, self.offsets = L, n_pairs, None

    def __getattr__(self, name):
        return getattr(self.L, name)

    def b200m_match_multiscale_batch(self, *a):
        a = list(a)
        a[11] = 1
        rc = self.L.b200m_match_multiscale_batch(*a)
        self.offsets = np.ctypeslib.as_array(a[12], shape=(self.n_pairs + 1,)).copy()
        return rc


@gpu
def test_wide_batch_errors_and_state():
    cases = [_case("fpfh", 2, 2, 100 + i, n_sk=400, n_tk=420) for i in range(3)]
    pairs, dim = [c[0] for c in cases], cases[0][3]
    with M.Context(0) as ctx:
        bad = [dict(p) for p in pairs]
        m = bad[1]["src_scales"][1][1].copy()
        m[5] = 400                                                # outside [0, n_src_kps)
        bad[1]["src_scales"] = [bad[1]["src_scales"][0], (bad[1]["src_scales"][1][0], m)]
        with pytest.raises(M.B200MatchError, match="pair 1, scale 1: an index map entry of the source"):
            ctx.match_wide_batch(2, M.MODE_MUTUAL, bad, dim)
        for mode in (M.MODE_RATIO, M.MODE_KNN_ONLY):
            with pytest.raises(M.B200MatchError, match="mode must be ONE_SIDED, MUTUAL or CLUSTER"):
                ctx.match_wide_batch(2, mode, pairs, dim)
        deep = [dict(p) for p in pairs]
        deep[2]["src_scales"] = deep[2]["src_scales"] * 3       # 6 scales
        deep[2]["tgt_scales"] = deep[2]["tgt_scales"] * 3
        with pytest.raises(M.B200MatchError, match=r"pair 2: n_scales \* k > 128"):
            ctx.match_wide_batch(32, M.MODE_MUTUAL, deep, dim)
        nox = [dict(p) for p in pairs]
        nox[1]["n_src_kps"] = len(nox[1]["src_kps_xyz"])
        nox[1]["src_kps_xyz"] = None
        with pytest.raises(M.B200MatchError, match="pair 1: null keypoint coordinates"):
            ctx.match_wide_batch(2, M.MODE_CLUSTER, nox, dim)
        one = ctx.match_wide_batch(2, M.MODE_ONE_SIDED, nox, dim)   # the one-sided matcher needs no source coordinates
        ref = ctx.match_wide_batch(2, M.MODE_ONE_SIDED, pairs, dim)
        assert all(a[0].tobytes() == b[0].tobytes() and a[1] == b[1] for a, b in zip(one, ref))
        offsets = np.zeros(1, np.uint64)
        p = M.Context._params(2, M.MODE_MUTUAL)
        rc = ctx._L.b200m_match_multiscale_batch(ctx._h, ctypes.byref(p), None, 0, 132, 33, 16, 40,
                                                 np.zeros(1, np.float32).ctypes.data, None, None, 0,
                                                 offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), None)
        assert rc != 0 and "give both threshold arrays or neither" in ctx._L.b200m_last_error(ctx._h).decode()
        L = ctx._L
        ctx._L = _CapOne(L, len(pairs))
        with pytest.raises(M.B200MatchError, match="capacity too small"):
            ctx.match_wide_batch(2, M.MODE_MUTUAL, pairs, dim)
        offs, ctx._L = ctx._L.offsets, L
        assert list(np.diff(offs.astype(np.int64))) == [len(r) for r, _ in ctx.match_wide_batch(2, M.MODE_MUTUAL, pairs, dim)]
        assert ctx.match_wide_batch(2, M.MODE_MUTUAL, [], dim) == []
        # single-pair calls on the same context after a batch
        with M.Context(0) as fresh:
            exp = _single(fresh, 2, M.MODE_CLUSTER, pairs[0], dim, cases[0][1], cases[0][2])
            s, t, _ = synth.make_pair("fpfh", 700, 800, seed=9)
            fresh.upload(0, s, 33)
            fresh.upload(1, t, 33)
            exp_m = fresh.match(2, M.MODE_MUTUAL)
        got = _single(ctx, 2, M.MODE_CLUSTER, pairs[0], dim, cases[0][1], cases[0][2])
        assert got[0].tobytes() == exp[0].tobytes() and got[1] == exp[1]
        ctx.match_wide_batch(2, M.MODE_MUTUAL, pairs, dim)
        ctx.upload(0, s, 33)
        ctx.upload(1, t, 33)
        got_m = ctx.match(2, M.MODE_MUTUAL)
        assert got_m[0].tobytes() == exp_m[0].tobytes() and got_m[1] == exp_m[1]


def _matchers(cls_id, k, n_scales, seeds, coords=True):
    out = []
    for i, seed in enumerate(seeds):
        pr, ts, tt, dim = _case("fpfh", k, n_scales, seed, n_sk=500 + 50 * i, n_tk=450 + 30 * i)
        rng = np.random.default_rng(seed)
        ks = rng.permutation(5 * len(pr["src_kps_xyz"]))[:len(pr["src_kps_xyz"])].astype(np.int32)
        kt = rng.permutation(5 * len(pr["tgt_kps_xyz"]))[:len(pr["tgt_kps_xyz"])].astype(np.int32)
        params = M.AlignmentParameters(randomness=k, distance_thr=float(DTHR), cluster_k=40, matching_id=cls_id)
        kw = dict(kps_xyz_src=pr["src_kps_xyz"], kps_xyz_tgt=pr["tgt_kps_xyz"], iss_radius_src=pr["iss_radius_src"],
                  iss_radius_tgt=pr["iss_radius_tgt"]) if coords else {}
        if i == 1:   # one matcher without thresholds in a batch with them
            ts = tt = None
        out.append(lambda pr=pr, ts=ts, tt=tt, dim=dim, ks=ks, kt=kt, params=params, kw=kw: M.get_feature_based_matcher_from_parameters(
            [a for a, _ in pr["src_scales"]], [a for a, _ in pr["tgt_scales"]], params, dim=dim, thresholds_src=ts,
            thresholds_tgt=tt, kps_indices_src=ks, kps_indices_tgt=kt,
            kps_indices_multiscale_src=[m for _, m in pr["src_scales"]], kps_indices_multiscale_tgt=[m for _, m in pr["tgt_scales"]],
            **kw))
    return out


@gpu
@pytest.mark.parametrize("cls_id,k,n_scales,coords", [(M.MATCHING_CLUSTER, 2, 2, True), (M.MATCHING_LEFT_TO_RIGHT, 3, 2, True),
                                                      (M.MATCHING_ONE_SIDED, 1, 1, True), (M.MATCHING_LEFT_TO_RIGHT, 1, 1, False),
                                                      (M.MATCHING_RATIO, 1, 1, False)],
                         ids=["cluster", "lr", "one_sided", "lr_identity_vote", "ratio"])
def test_match_many_equals_match(cls_id, k, n_scales, coords):
    makers = _matchers(cls_id, k, n_scales, [110, 111, 112, 113], coords)
    ref = []
    for mk in makers:
        m = mk()
        ref.append((m.match(), m.get_average_distance()))
    ms = [mk() for mk in makers]
    if not coords:   # one candidate per keypoint and no coordinates: the k-list route (match_batch)
        assert all(isinstance(m, M.RatioMatcher) or not m._uses_wide_seam() for m in ms)
    got = M.match_many(ms)
    for m, g, (r, ravg) in zip(ms, got, ref):
        assert g.tobytes() == r.tobytes() and m.get_average_distance() == ravg
    assert sum(len(g) for g in got) > 0


@gpu
def test_match_many_rejects_mixed_matchers():
    a = _matchers(M.MATCHING_CLUSTER, 2, 2, [120])[0]()
    b = _matchers(M.MATCHING_LEFT_TO_RIGHT, 2, 2, [121])[0]()
    c = _matchers(M.MATCHING_CLUSTER, 2, 2, [122])[0]()
    c.parameters = M.AlignmentParameters(randomness=2, cluster_k=20, matching_id=M.MATCHING_CLUSTER)
    with pytest.raises(M.B200MatchError, match="one class"):
        M.match_many([a, b])
    with pytest.raises(M.B200MatchError, match="one class"):
        M.match_many([a, c])
    assert M.match_many([]) == []


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "lr", "cluster"])
def test_cpp_wide_batch_program_matches_oracle(tmp_path, mode):
    exe = _build_exe()
    k = 2
    cases = [_case("fpfh", k, 2, 130, n_sk=600, n_tk=650), _case("fpfh", k, 1, 131, n_sk=300, n_tk=257, identity=False),
             _case("fpfh", k, 3, 132, n_sk=450, n_tk=500)]
    blob = bytearray()
    for pr, _, _, _ in cases:
        ns, nt = len(pr["src_kps_xyz"]), len(pr["tgt_kps_xyz"])
        blob += np.array([len(pr["src_scales"]), ns, nt], np.int32).tobytes()
        blob += np.array([pr["iss_radius_src"], pr["iss_radius_tgt"]], np.float32).tobytes()
        for (sf, sm), (tf, tm) in zip(pr["src_scales"], pr["tgt_scales"]):
            blob += np.array([len(sf), len(tf)], np.int32).tobytes()
            for f, m, n in ((sf, sm, ns), (tf, tm, nt)):
                blob += np.ascontiguousarray(f, np.float32).tobytes()
                blob += (np.arange(len(f), dtype=np.int32) if m is None else m).tobytes()
        blob += pr["src_kps_xyz"].tobytes() + pr["tgt_kps_xyz"].tobytes()
    bp, op = tmp_path / "pairs.bin", tmp_path / "o.txt"
    bp.write_bytes(bytes(blob))
    r = subprocess.run([exe, mode, str(k), str(bp), str(len(cases)), str(op)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    head, corr = {}, {}
    for line in open(op):
        w = line.split()
        if w[0] == "pair":
            head[int(w[1])] = (int(w[2]), np.float32(w[3]), int(w[4]))
        elif w[0] == "corr":
            corr.setdefault(int(w[1]), []).append((int(w[2]), int(w[3]), np.float32(w[4]), np.float32(w[5])))
    oname = {"one_sided": "one_sided", "lr": "mutual", "cluster": "cluster"}[mode]
    for p, (pr, _, _, _) in enumerate(cases):
        e, eavg = orc.match_wide(oname, pr["src_scales"], pr["tgt_scales"], pr["src_kps_xyz"][:, :3], pr["tgt_kps_xyz"][:, :3],
                                 pr["iss_radius_src"], pr["iss_radius_tgt"], k, 40, np.float32(M.FLT_MAX))
        n, avg, same = head[p]
        assert same == 1 and n == len(e) and avg == np.float32(eavg)
        assert corr.get(p, []) == [(int(a), int(b), np.float32(c), np.float32(d)) for a, b, c, d in
                                   zip(e["index_query"], e["index_match"], e["distance"], e["threshold"])]
