"""b200m_match_multiscale_local_batch (Context.match_wide_local_batch, guessed matchers, match_many, b200match::matchMany):
the matcher classes at the wide seam with AlignmentParameters::guess set.  Records and averages must equal, byte for byte,
the oracle's guessed composition (matchLocal per scale and direction, then the vote and the filter), which is itself
checked against a literal Python-loop restatement.  The GPU tests run with -m gpu on a B200; the rest need none."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from lidar_global_registration_b200 import build as b200_build
from lidar_global_registration_b200 import matcher as M
from oracle import oracle as orc
from test_gpu_wide_batch import DTHR, GMODE, _case, _edge_cases, _xyz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "wide_local_test")
gpu = pytest.mark.gpu
FLT_MAX = np.float32(M.FLT_MAX)


# ---- the oracle's guessed composition -------------------------------------------------------------------------------------
def _rows_xyz(xyz, kp_map, n):
    x = np.asarray(xyz, np.float32)[:, :3]
    return np.ascontiguousarray(x[:n] if kp_map is None else x[np.asarray(kp_map, np.int64)])


def oracle_match_multiscale_local(query_scales, train_scales, n_query_kps, query_moved, train_xyz, iss_radius, k, radius):
    """match_multiscale with a guess (include/matching.h:297-311): per scale orc.match_local over that scale's rows, the
    query rows at their MOVED keypoints, the train rows at their keypoints; then match_multiscale's remap, concatenation and
    vote over the unmoved train keypoints."""
    comb_i = [[] for _ in range(n_query_kps)]
    comb_d = [[] for _ in range(n_query_kps)]
    for (qf, qmap), (tf, tmap) in zip(query_scales, train_scales):
        if qf.shape[0] == 0:
            continue
        ei, ed, ec = orc.match_local(qf, tf, k, _rows_xyz(query_moved, qmap, len(qf)), _rows_xyz(train_xyz, tmap, len(tf)),
                                     np.float32(radius))
        for r in range(qf.shape[0]):
            kp = r if qmap is None else int(qmap[r])
            for m in range(ec[r]):
                j = int(ei[r, m])
                comb_i[kp].append(j if tmap is None else int(tmap[j]))
                comb_d[kp].append(ed[r, m])
    return _vote(comb_i, comb_d, train_xyz, iss_radius)


def _vote(comb_i, comb_d, train_xyz, iss_radius):
    n = len(comb_i)
    width = max(max((len(c) for c in comb_i), default=0), 1)
    ci, cd, cc = np.full((n, width), -1, np.int32), np.zeros((n, width), np.float32), np.zeros(n, np.int32)
    for i in range(n):
        cc[i] = len(comb_i[i])
        ci[i, :cc[i]] = comb_i[i]
        cd[i, :cc[i]] = comb_d[i]
    xyz = np.ascontiguousarray(np.asarray(train_xyz, np.float32)[:, :3])
    if xyz.shape[0] == 0:
        return ci[:, :1].copy(), cd[:, :1].copy(), np.zeros(n, np.int32)
    vi, vd, vc = orc.spatial_vote(ci, cd, cc, xyz, iss_radius)
    return np.ascontiguousarray(vi[:, :1]), np.ascontiguousarray(vd[:, :1]), vc


def _filter(mode, fwd, rev, src_xyz, tgt_xyz, cluster_k, distance_thr, thr_q, thr_t):
    fi, fd, fc = fwd
    avg = orc.average_distance(fd, fc)
    if mode == "one_sided":
        return orc.filter_one_sided(fi, fd, fc, distance_thr, thr_q, thr_t), avg
    ri, rd, rc = rev
    if mode == "mutual":
        return orc.filter_mutual(fi, fc, ri, rd, rc, distance_thr, thr_q, thr_t), avg
    if len(src_xyz) == 0 or len(tgt_xyz) == 0:
        return np.empty(0, orc.CORR_DTYPE), avg
    return orc.filter_cluster(fi, fc, ri, rc, orc.knn3d(src_xyz, cluster_k), orc.knn3d(tgt_xyz, cluster_k), distance_thr,
                              thr_q=thr_q, thr_t=thr_t), avg


def oracle_match_wide_local(mode, pr, k, radius, cluster_k=40, distance_thr=DTHR, thr_q=None, thr_t=None):
    """match_impl with a guess: `pr` is a match_wide_local_batch pair (src/tgt_kps_moved given)"""
    sx, tx = pr["src_kps_xyz"][:, :3], pr["tgt_kps_xyz"][:, :3]
    fwd = oracle_match_multiscale_local(pr["src_scales"], pr["tgt_scales"], len(sx), pr["src_kps_moved"], tx, pr["iss_radius_tgt"],
                                        k, radius)
    rev = None if mode == "one_sided" else oracle_match_multiscale_local(
        pr["tgt_scales"], pr["src_scales"], len(tx), pr["tgt_kps_moved"], sx, pr["iss_radius_src"], k, radius)
    return _filter(mode, fwd, rev, sx, tx, cluster_k, distance_thr, thr_q, thr_t)


# ---- a literal restatement of the gated kNN, for the oracle's composition ------------------------------------------------------
def _loop_multiscale_local(query_scales, train_scales, n_query_kps, query_moved, train_xyz, iss_radius, k, radius):
    r2 = np.float32(radius) * np.float32(radius)
    comb_i = [[] for _ in range(n_query_kps)]
    comb_d = [[] for _ in range(n_query_kps)]
    for (qf, qmap), (tf, tmap) in zip(query_scales, train_scales):
        for r in range(len(qf)):
            kp = r if qmap is None else int(qmap[r])
            if not np.all(np.isfinite(qf[r])):
                continue
            a = np.asarray(query_moved, np.float32)[kp, :3]
            hits = []
            for j in range(len(tf)):
                b = np.asarray(train_xyz, np.float32)[j if tmap is None else int(tmap[j]), :3]
                d = [np.float32(a[c] - b[c]) for c in range(3)]
                s = np.float32(np.float32(np.float32(d[0] * d[0]) + np.float32(d[1] * d[1])) + np.float32(d[2] * d[2]))
                if s < r2 and np.all(np.isfinite(tf[j])):
                    hits.append((np.float32(orc.l2_norm(qf[r], tf[j])), s, j))
            for dd, _, j in sorted(hits)[:k]:
                comb_i[kp].append(j if tmap is None else int(tmap[j]))
                comb_d[kp].append(dd)
    return _vote(comb_i, comb_d, train_xyz, iss_radius)


def _loop_match_wide_local(mode, pr, k, radius, cluster_k):
    sx, tx = pr["src_kps_xyz"][:, :3], pr["tgt_kps_xyz"][:, :3]
    fwd = _loop_multiscale_local(pr["src_scales"], pr["tgt_scales"], len(sx), pr["src_kps_moved"], tx, pr["iss_radius_tgt"], k,
                                 radius)
    rev = None if mode == "one_sided" else _loop_multiscale_local(
        pr["tgt_scales"], pr["src_scales"], len(tx), pr["tgt_kps_moved"], sx, pr["iss_radius_src"], k, radius)
    return _filter(mode, fwd, rev, sx, tx, cluster_k, DTHR, None, None)


def _rigid(seed, angle=0.2, shift=0.3):
    """a rigid guess (rotation about a random axis, a translation) as 16 floats, row-major"""
    rng = np.random.default_rng(seed)
    ax = rng.standard_normal(3)
    ax /= np.linalg.norm(ax)
    t = angle * rng.random()
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    g = np.eye(4)
    g[:3, :3] = np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K
    g[:3, 3] = shift * rng.standard_normal(3)
    return tuple(float(v) for v in g.astype(np.float32).ravel())


def _guessed(pr, guess):
    pr = dict(pr)
    pr["src_kps_moved"] = M.transform_keypoints(pr["src_kps_xyz"], guess)
    pr["tgt_kps_moved"] = M.transform_keypoints(pr["tgt_kps_xyz"], M.invert_guess(guess))
    return pr


# ---- without a GPU ------------------------------------------------------------------------------------------------------
def test_local_pair_struct_is_the_c_layout(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "b200match.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(b200m_local_pair));\n' +
                   "".join('  printf(" %%zu", offsetof(b200m_local_pair, %s));\n' % n for n, _ in M._LocalPair._fields_) +
                   '  printf("\\n");\n  (void) b200m_match_multiscale_local_batch;\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [ctypes.sizeof(M._LocalPair)] + [getattr(M._LocalPair, n).offset for n, _ in M._LocalPair._fields_]
    assert "b200m_match_multiscale_local_batch" in M.EXPORTS


def test_transform_keypoints_order_and_inverse_round_trip():
    rng = np.random.default_rng(1)
    x = (rng.random((500, 4)) * 40 - 20).astype(np.float32)
    g = _rigid(7, angle=1.0, shift=5.0)
    got = M.transform_keypoints(x, g)
    G = np.asarray(g, np.float32).reshape(4, 4)
    for i in range(0, 500, 37):
        for r in range(3):
            e = np.float32(np.float32(np.float32(G[r, 0] * x[i, 0]) + np.float32(G[r, 1] * x[i, 1])) + np.float32(G[r, 2] * x[i, 2]))
            assert got[i, r] == np.float32(e + G[r, 3])
    assert np.array_equal(got[:, 3], x[:, 3])
    back = M.transform_keypoints(got, M.invert_guess(g))
    ulp = np.spacing(np.maximum(np.abs(x[:, :3]), 20).astype(np.float32))
    assert np.all(np.abs(back[:, :3] - x[:, :3]) <= 8 * ulp)
    assert np.allclose(M.invert_guess(M.invert_guess(g)), G, atol=1e-6)


def _small_pair(seed, nan=False):
    """integer keypoints, so that some train keypoints lie exactly at distance 2 (= the radius: excluded), descriptors with
    exact ties (duplicated rows), NaN coordinates on request"""
    rng = np.random.default_rng(seed)
    sx = np.zeros((14, 4), np.float32)
    tx = np.zeros((16, 4), np.float32)
    sx[:, :3] = rng.integers(0, 5, (14, 3))
    tx[:, :3] = rng.integers(0, 5, (16, 3))
    if nan:
        sx[3, 0] = np.nan
        tx[5, 1] = np.nan
    s_sc, t_sc = [], []
    for s, (ns, nt) in enumerate([(14, 16), (10, 12)]):
        sf = rng.integers(0, 3, (ns, 33)).astype(np.float32)
        tf = rng.integers(0, 3, (nt, 33)).astype(np.float32)
        tf[1] = tf[0]
        tf[7] = tf[4]
        sf[2] = tf[0]
        smap = None if s == 0 else np.sort(rng.choice(14, ns, replace=False)).astype(np.int32)
        tmap = None if s == 0 else np.sort(rng.choice(16, nt, replace=False)).astype(np.int32)
        s_sc.append((sf, smap))
        t_sc.append((tf, tmap))
    g = (1, 0, 0, 1, 0, 1, 0, 0, 0, 0, 1, -1, 0, 0, 0, 1)   # an integer shift: distances stay integers
    return _guessed(dict(src_scales=s_sc, tgt_scales=t_sc, src_kps_xyz=sx, tgt_kps_xyz=tx, iss_radius_src=np.float32(1.5),
                         iss_radius_tgt=np.float32(1.5)), g)


@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
@pytest.mark.parametrize("nan", [False, True])
def test_oracle_guessed_composition_equals_python_loops(mode, nan):
    for seed in range(3):
        pr = _small_pair(seed, nan)
        for k, radius in ((1, 2.0), (3, 2.0), (2, 3.5)):
            e, eavg = oracle_match_wide_local(mode, pr, k, radius, cluster_k=4)
            lo, lavg = _loop_match_wide_local(mode, pr, k, radius, cluster_k=4)
            assert e.tobytes() == lo.tobytes() and eavg == lavg
    # the vote inputs themselves, per direction: the gated lists of the loops equal orc.match_local's
    pr = _small_pair(5, nan)
    a = oracle_match_multiscale_local(pr["src_scales"], pr["tgt_scales"], 14, pr["src_kps_moved"], pr["tgt_kps_xyz"], 1.5, 3, 2.0)
    b = _loop_multiscale_local(pr["src_scales"], pr["tgt_scales"], 14, pr["src_kps_moved"], pr["tgt_kps_xyz"], 1.5, 3, 2.0)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))


def test_gate_excludes_distance_equal_to_radius():
    pr = _small_pair(2)
    fwd = _loop_multiscale_local(pr["src_scales"][:1], pr["tgt_scales"][:1], 14, pr["src_kps_moved"], pr["tgt_kps_xyz"], 0.0, 16, 2.0)
    mv, tx = pr["src_kps_moved"][:, :3], pr["tgt_kps_xyz"][:, :3]
    at_r = [(i, j) for i in range(14) for j in range(16) if np.sum((mv[i] - tx[j]) ** 2) == 4]
    assert at_r   # the case exists
    ei, _, ec = orc.match_local(pr["src_scales"][0][0], pr["tgt_scales"][0][0], 16, mv, tx, np.float32(2.0))
    for i, j in at_r:
        assert j not in ei[i, :ec[i]]
    assert fwd[0].shape[0] == 14


def _matcher(cls, guess=None, coords=True, **kw):
    pr, ts, tt, dim = _case("fpfh", 2, 2, 3, n_sk=300, n_tk=320)
    params = M.AlignmentParameters(randomness=2, cluster_k=40, matching_id=cls, guess=guess, **kw)
    xyz = dict(kps_xyz_src=pr["src_kps_xyz"], kps_xyz_tgt=pr["tgt_kps_xyz"], iss_radius_src=pr["iss_radius_src"],
               iss_radius_tgt=pr["iss_radius_tgt"]) if coords else {}
    return M.get_feature_based_matcher_from_parameters(
        [a for a, _ in pr["src_scales"]], [a for a, _ in pr["tgt_scales"]], params, dim=dim,
        kps_indices_multiscale_src=[m for _, m in pr["src_scales"]], kps_indices_multiscale_tgt=[m for _, m in pr["tgt_scales"]],
        **xyz)


def test_guess_refusals_come_before_the_device(monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("a device was used")
    monkeypatch.setattr(M, "Context", no_device)
    g = _rigid(1)
    with pytest.raises(M.B200MatchError, match="RatioMatcher: a guess is not supported"):
        _matcher(M.MATCHING_RATIO, g).match()
    with pytest.raises(M.B200MatchError, match="a guess needs kps_xyz_src/tgt"):
        _matcher(M.MATCHING_LEFT_TO_RIGHT, g, coords=False).match()
    with pytest.raises(M.B200MatchError, match="a guess or none"):
        M.match_many([_matcher(M.MATCHING_LEFT_TO_RIGHT, g), _matcher(M.MATCHING_LEFT_TO_RIGHT)])
    with pytest.raises(M.B200MatchError, match="RatioMatcher: a guess is not supported"):
        M.match_many([_matcher(M.MATCHING_RATIO, g), _matcher(M.MATCHING_RATIO, _rigid(2))])
    # the guess is not part of the comparison, every other field is
    with pytest.raises(M.B200MatchError, match="one class"):
        M.match_many([_matcher(M.MATCHING_LEFT_TO_RIGHT, g), _matcher(M.MATCHING_LEFT_TO_RIGHT, g, match_search_radius=1.0)])
    assert M.AlignmentParameters(guess=g) == M.AlignmentParameters(guess=tuple(g))


def _build_exe():
    b200_build.build()
    src = os.path.join(ROOT, "tests", "cpp", "wide_local_test.cpp")
    deps = [src, os.path.join(ROOT, "include", "b200match_shim.hpp"), os.path.join(ROOT, "include", "b200match.h")]
    if os.path.exists(EXE) and all(os.path.getmtime(EXE) >= os.path.getmtime(d) for d in deps):
        return EXE
    libdir = os.path.join(ROOT, "lidar_global_registration_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                    "-L", libdir, "-l:libb200match.so", "-Wl,-rpath," + libdir], check=True)
    return EXE


def test_wide_local_program_compiles_and_links():
    r = subprocess.run([_build_exe()], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


# ---- on the GPU -----------------------------------------------------------------------------------------------------------
def _check(mode, k, cases, radius, guesses):
    pairs = [_guessed(c[0], g) for c, g in zip(cases, guesses)]
    ts, tt = [c[1] for c in cases], [c[2] for c in cases]
    with M.Context(0) as ctx:
        got = ctx.match_wide_local_batch(k, GMODE[mode], pairs, radius, cases[0][3], 40, DTHR, ts, tt)
    assert len(got) == len(pairs)
    for p, (recs, avg) in enumerate(got):
        pr = pairs[p]
        if not pr["src_scales"] or not len(pr["src_kps_xyz"]):
            assert len(recs) == 0 and avg == M.FLT_MAX
            continue
        e, eavg = oracle_match_wide_local(mode, pr, k, radius, 40, DTHR, ts[p], tt[p])
        assert recs.tobytes() == e.tobytes() and avg == np.float32(eavg), (mode, p)
    return got


COMBOS = [("fpfh", 1, 1), ("fpfh", 2, 1), ("shot", 2, 2), ("rops", 3, 3), ("fpfh", 5, 2)]


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
@pytest.mark.parametrize("desc,k,n_scales", COMBOS)
def test_wide_local_equals_oracle(desc, k, n_scales, mode):
    cases = [_case(desc, k, n_scales, 31 + 7 * k + n_scales), _case(desc, k, n_scales, 5, n_sk=300, n_tk=420),
             _case(desc, k, n_scales, 6, n_sk=600, n_tk=257, identity=False)]
    got = _check(mode, k, cases, 0.6, [_rigid(10 + i, 0.05, 0.05) for i in range(3)])
    assert sum(len(r) for r, _ in got) > 0


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
@pytest.mark.parametrize("radius", [0.25, 1.5, 10.0, float(FLT_MAX), float("inf")], ids=["many_cells", "few_cells", "whole_cloud",
                                                                                          "flt_max", "inf"])
def test_wide_local_radii(mode, radius):
    cases = [_case("fpfh", 2, 2, 20 + i, n_sk=700 - 100 * i, n_tk=650) for i in range(3)]
    _check(mode, 2, cases, radius, [_rigid(20 + i, 0.1, 0.1) for i in range(3)])


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
def test_wide_local_edge_cases(mode):
    cases = _edge_cases(2)
    cases[7][0]["src_scales"][1][0][:, :] = np.nan
    if mode != "cluster":   # NaN keypoints on both sides (the cluster filter's 3-D neighbourhoods of NaN points are not pinned)
        cases[0][0]["src_kps_xyz"][::7, 1] = np.nan
        cases[9][0]["tgt_kps_xyz"][::11, 2] = np.nan
    guesses = [_rigid(40 + i, 0.1, 0.1) for i in range(len(cases))]
    guesses[1] = (1, 0, 0, 100, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1)   # the source moved out of the target's box
    got = _check(mode, 2, cases, 0.8, guesses)
    assert len(got[1][0]) == 0
    assert len(got[3][0]) == 0 and got[3][1] == M.FLT_MAX and len(got[8][0]) == 0
    got0 = _check(mode, 2, cases, 0.0, guesses)          # radius 0: nothing passes the gate
    assert all(len(r) == 0 for r, _ in got0)
    _check(mode, 2, cases, float("nan"), guesses)


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
def test_wide_local_pairs_stay_isolated(mode):
    """identical coordinates in every pair, a different guess each: a cell that leaked across pairs would change a result;
    then two pairs swap their guesses"""
    rng = np.random.default_rng(3)
    sx, tx = _xyz(rng, 600), _xyz(rng, 640)
    cases = [_case("fpfh", 2, 2, 60 + i, n_sk=600, n_tk=640, sx=sx, tx=tx) for i in range(4)]
    guesses = [_rigid(60 + i, 0.3, 0.4) for i in range(4)]
    _check(mode, 2, cases, 0.5, guesses)
    guesses[0], guesses[2] = guesses[2], guesses[0]
    _check(mode, 2, cases, 0.5, guesses)


@gpu
def test_wide_local_launch_count_does_not_grow_with_pairs():
    launches = []
    for n in (2, 32):
        cases = [_case("fpfh", 2, 2, 70, n_sk=300, n_tk=300)] * n
        pairs = [_guessed(c[0], _rigid(70)) for c in cases]
        with M.Context(0) as ctx:
            ctx.set_profiling(True)
            ctx.reset_stats()
            ctx.match_wide_local_batch(2, M.MODE_CLUSTER, pairs, 0.5, cases[0][3])
            launches.append(ctx.stats()["launches"])
    assert launches[0] == launches[1], launches


@gpu
def test_wide_local_errors_and_state():
    cases = [_case("fpfh", 2, 2, 100 + i, n_sk=400, n_tk=420) for i in range(3)]
    pairs, dim = [_guessed(c[0], _rigid(100 + i)) for i, c in enumerate(cases)], cases[0][3]
    with M.Context(0) as ctx:
        bad = [dict(p) for p in pairs]
        bad[2]["tgt_kps_moved"] = None
        with pytest.raises(M.B200MatchError, match="pair 2: null moved keypoint coordinates"):
            ctx.match_wide_local_batch(2, M.MODE_MUTUAL, bad, 0.5, dim)
        one = ctx.match_wide_local_batch(2, M.MODE_ONE_SIDED, bad, 0.5, dim)   # the one-sided matcher has no reverse pass
        ref = ctx.match_wide_local_batch(2, M.MODE_ONE_SIDED, pairs, 0.5, dim)
        assert all(a[0].tobytes() == b[0].tobytes() and a[1] == b[1] for a, b in zip(one, ref))
        bad = [dict(p) for p in pairs]
        m = bad[1]["tgt_scales"][1][1].copy()
        m[3] = -1
        bad[1]["tgt_scales"] = [bad[1]["tgt_scales"][0], (bad[1]["tgt_scales"][1][0], m)]
        with pytest.raises(M.B200MatchError, match="b200m_match_multiscale_local_batch: pair 1, scale 1: an index map entry of the target"):
            ctx.match_wide_local_batch(2, M.MODE_MUTUAL, bad, 0.5, dim)
        offsets = np.zeros(2, np.uint64)
        p = M.Context._params(2, M.MODE_MUTUAL)
        arr = (M._WidePair * 1)()
        rc = ctx._L.b200m_match_multiscale_local_batch(ctx._h, ctypes.byref(p), arr, None, 1, 132, 33, 16, 40, 0.5, None, None,
                                                       None, 0, offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), None)
        assert rc != 0 and "null local pairs" in ctx._L.b200m_last_error(ctx._h).decode()
        L = ctx._L

        class CapOne:
            def __getattr__(self, name):
                return getattr(L, name)

            def b200m_match_multiscale_local_batch(self, *a):
                a = list(a)
                a[13] = 1
                rc = L.b200m_match_multiscale_local_batch(*a)
                self.offsets = np.ctypeslib.as_array(a[14], shape=(len(pairs) + 1,)).copy()
                return rc
        ctx._L = CapOne()
        with pytest.raises(M.B200MatchError, match="capacity too small"):
            ctx.match_wide_local_batch(2, M.MODE_MUTUAL, pairs, 0.5, dim)
        offs, ctx._L = ctx._L.offsets, L
        full = ctx.match_wide_local_batch(2, M.MODE_MUTUAL, pairs, 0.5, dim)
        assert list(np.diff(offs.astype(np.int64))) == [len(r) for r, _ in full]
        # the unguessed batch and the single-pair calls on the same context afterwards
        with M.Context(0) as fresh:
            exp = fresh.match_wide_batch(2, M.MODE_CLUSTER, [c[0] for c in cases], dim)
        got = ctx.match_wide_batch(2, M.MODE_CLUSTER, [c[0] for c in cases], dim)
        assert all(a[0].tobytes() == b[0].tobytes() and a[1] == b[1] for a, b in zip(got, exp))
        again = ctx.match_wide_local_batch(2, M.MODE_MUTUAL, pairs, 0.5, dim)
        assert all(a[0].tobytes() == b[0].tobytes() and a[1] == b[1] for a, b in zip(again, full))


@gpu
@pytest.mark.parametrize("cls_id", [M.MATCHING_CLUSTER, M.MATCHING_LEFT_TO_RIGHT, M.MATCHING_ONE_SIDED])
def test_guessed_match_equals_match_many_and_oracle(cls_id):
    ms, ref = [], []
    for i in range(3):
        m = _matcher(cls_id, _rigid(110 + i, 0.1, 0.1), match_search_radius=0.6, distance_thr=float(DTHR))
        m.src = [a.copy() for a in m.src]
        ms.append(m)
        ref.append((m.match(), m.get_average_distance()))
    got = M.match_many(ms)
    mode = {M.MATCHING_CLUSTER: "cluster", M.MATCHING_LEFT_TO_RIGHT: "mutual", M.MATCHING_ONE_SIDED: "one_sided"}[cls_id]
    for m, g, (r, ravg) in zip(ms, got, ref):
        assert g.tobytes() == r.tobytes() and m.get_average_distance() == ravg
        e, eavg = oracle_match_wide_local(mode, _guessed(m._wide_pair(), m.parameters.guess), 2, 0.6)
        assert r.tobytes() == e.tobytes() and ravg == np.float32(eavg)
    assert sum(len(g) for g in got) > 0


@gpu
def test_wide_local_full_size():
    cases = [_case("fpfh", 2, 3, 200 + i, n_sk=20000, n_tk=20000) for i in range(4)]
    got = _check("mutual", 2, cases, 0.15, [_rigid(200 + i, 0.02, 0.02) for i in range(4)])
    assert sum(len(r) for r, _ in got) > 0


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "lr", "cluster"])
def test_cpp_wide_local_program_matches_oracle(tmp_path, mode):
    exe = _build_exe()
    k, radius = 2, np.float32(0.6)
    cases = [_case("fpfh", k, 2, 130, n_sk=600, n_tk=650), _case("fpfh", k, 1, 131, n_sk=300, n_tk=257, identity=False),
             _case("fpfh", k, 3, 132, n_sk=450, n_tk=500)]
    guesses = [_rigid(130 + i, 0.1, 0.1) for i in range(3)]
    blob = bytearray()
    for (pr, _, _, _), g in zip(cases, guesses):
        ns, nt = len(pr["src_kps_xyz"]), len(pr["tgt_kps_xyz"])
        blob += np.array([len(pr["src_scales"]), ns, nt], np.int32).tobytes()
        blob += np.array([pr["iss_radius_src"], pr["iss_radius_tgt"]], np.float32).tobytes()
        blob += np.array(g, np.float32).tobytes()
        for (sf, sm), (tf, tm) in zip(pr["src_scales"], pr["tgt_scales"]):
            blob += np.array([len(sf), len(tf)], np.int32).tobytes()
            for f, m in ((sf, sm), (tf, tm)):
                blob += np.ascontiguousarray(f, np.float32).tobytes()
                blob += (np.arange(len(f), dtype=np.int32) if m is None else m).tobytes()
        blob += pr["src_kps_xyz"].tobytes() + pr["tgt_kps_xyz"].tobytes()
    bp, op = tmp_path / "pairs.bin", tmp_path / "o.txt"
    bp.write_bytes(bytes(blob))
    r = subprocess.run([exe, mode, str(k), str(bp), str(len(cases)), repr(float(radius)), str(op)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    head, corr = {}, {}
    for line in open(op):
        w = line.split()
        if w[0] == "pair":
            head[int(w[1])] = (int(w[2]), np.float32(w[3]), int(w[4]))
        elif w[0] == "corr":
            corr.setdefault(int(w[1]), []).append((int(w[2]), int(w[3]), np.float32(w[4]), np.float32(w[5])))
    moved = np.fromfile(str(op) + ".moved", np.float32)
    oname = {"one_sided": "one_sided", "lr": "mutual", "cluster": "cluster"}[mode]
    at = 0
    for p, (pr, _, _, _) in enumerate(cases):
        pr = dict(pr)
        for side, n in (("src_kps_moved", len(pr["src_kps_xyz"])), ("tgt_kps_moved", len(pr["tgt_kps_xyz"]))):
            pr[side] = moved[at:at + 4 * n].reshape(n, 4)   # the coordinates the shim moved, as it moved them
            at += 4 * n
        e, eavg = oracle_match_wide_local(oname, pr, k, radius, 40, FLT_MAX)
        n, avg, same = head[p]
        assert same == 1 and n == len(e) and avg == np.float32(eavg)
        assert corr.get(p, []) == [(int(a), int(b), np.float32(c), np.float32(d)) for a, b, c, d in
                                   zip(e["index_query"], e["index_match"], e["distance"], e["threshold"])]
