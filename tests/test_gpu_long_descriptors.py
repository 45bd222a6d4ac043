"""Descriptors longer than 637 floats: the K-streamed tensor-core pass (640 < kp <= 2048, i.e. dim <= 2045) and the exact
path for dim 2046..2048, up to USC-1960 (pcl::UniqueShapeContext1960, 7876-byte rows).  Every result is compared byte for
byte with the oracle, or, for device calls, with their host form.  The generator's layout and the C++ program's build are
checked without a GPU."""
import os
import subprocess

import numpy as np
import pytest

from lidar_global_registration_b200 import build as b200_build
from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "usc_test")
gpu = pytest.mark.gpu
USC_DIM, USC_STRIDE = synth.DESCRIPTORS["usc"]

DIMS = [638, 700, 1000, 1021, 1022, 1024, 1025, 1500, 1960, 1981, 2045, 2046, 2048]
KINDS = ["uniform", "clustered", "duplicates", "offset", "tiny", "huge", "sparse", "integers", "near_ties"]
KS = [1, 2, 5, 16]


def _dense(a, dim):
    return np.ascontiguousarray(a[:, :dim])


def _same(got, exp):
    for a, b in zip(got, exp):
        assert np.array_equal(a, b)


# ---- without a GPU ----------------------------------------------------------------------------------------------------------
def test_usc_generator_layout():
    src, tgt, dim = synth.make_pair("usc", 500, 640, nan_frac=0.01)
    assert (dim, USC_STRIDE) == (1960, 1969)
    for a in (src, tgt):
        assert a.dtype == np.float32 and a.shape[1] == 1969
        assert np.isfinite(a[:, dim:]).all()                        # the rf[9] tail: junk, but finite
        bad = ~np.isfinite(a[:, :dim]).all(1)
        assert bad.sum() == int(round(0.01 * a.shape[0]))           # nan_frac rows carry one NaN
        assert a[~bad, :dim].min() >= 0                              # non-negative
    assert (src[:, :USC_DIM] == 0).mean() > 0.6                      # the generator's rows are mostly zero (the target's
                                                                     # copies carry dense noise)
    # clustered around prototypes: the nearest other source row is much closer than a random one
    s = src[np.isfinite(src[:, :dim]).all(1), :dim].astype(np.float64)[:200]
    d2 = ((s[:, None, :] - s[None, :, :]) ** 2).sum(-1)
    np.fill_diagonal(d2, np.inf)
    assert np.median(d2.min(1)) < 0.5 * np.median(d2[np.isfinite(d2)])


def _build_exe():
    b200_build.build()
    src = os.path.join(ROOT, "tests", "cpp", "usc_test.cpp")
    deps = [src, os.path.join(ROOT, "include", "b200match_shim.hpp"), os.path.join(ROOT, "include", "b200match.h")]
    if os.path.exists(EXE) and all(os.path.getmtime(EXE) >= os.path.getmtime(d) for d in deps):
        return EXE
    libdir = os.path.join(ROOT, "lidar_global_registration_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                    "-L", libdir, "-l:libb200match.so", "-Wl,-rpath," + libdir], check=True)
    return EXE


def test_usc_program_compiles_and_links():
    """tests/cpp/usc_test.cpp builds against the shim (its static_assert pins sizeof(UniqueShapeContext1960) == 7876)"""
    r = subprocess.run([_build_exe()], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


# ---- on the GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def _built():
    b200_build.build()
    M.load_library()


def _make(rng, kind, n, dim):
    # the data kinds of test_gpu_fuzz.py
    if kind == "uniform":
        a = rng.random((n, dim))
    elif kind == "clustered":
        protos = rng.random((max(n // 40, 2), dim))
        a = protos[rng.integers(0, protos.shape[0], n)] + 0.01 * rng.standard_normal((n, dim))
    elif kind == "duplicates":
        base = rng.random((max(n // 5, 1), dim))
        a = base[rng.integers(0, base.shape[0], n)]
    elif kind == "offset":
        a = 1e4 + rng.random((n, dim))
    elif kind == "tiny":
        a = 1e-32 * rng.random((n, dim))
    elif kind == "huge":
        a = 1e32 * rng.random((n, dim))
    elif kind == "near_ties":
        base = rng.random((max(n // 200, 1), dim))
        a = base[rng.integers(0, base.shape[0], n)] + 1e-6 * rng.standard_normal((n, dim))
    elif kind == "sparse":
        a = rng.random((n, dim)) * (rng.random((n, dim)) < 0.2)
    else:
        a = rng.integers(0, 3, (n, dim)).astype(np.float64)
    return a.astype(np.float32)


def _case(seed):
    rng = np.random.default_rng(7000 + seed)
    dim = DIMS[seed % len(DIMS)]
    kind = KINDS[(seed // 2) % len(KINDS)]
    k = KS[(seed // 3) % len(KS)]
    nq = int(rng.choice([1, 127, 129, 300, 600]))
    nt = int(rng.choice([5, 255, 257, 513, 900]))
    stride = dim + int(rng.choice([0, 1, 9]))              # AoS with a junk tail
    q = np.zeros((nq, stride), np.float32)
    t = np.zeros((nt, stride), np.float32)
    both = _make(rng, kind, nq + nt, dim)
    q[:, :dim], t[:, :dim] = both[:nq], both[nq:]
    q[:, dim:] = np.nan
    t[:, dim:] = np.inf
    for a in (q, t):                                       # NaN / Inf rows
        bad = rng.random(a.shape[0]) < 0.03
        a[bad, rng.integers(0, dim)] = rng.choice([np.nan, np.inf, -np.inf])
    return q, t, dim, k, kind


@gpu
@pytest.mark.parametrize("seed", range(52))
def test_long_knn_fuzz(_built, seed):
    q, t, dim, k, kind = _case(seed)
    with M.Context(0) as ctx:
        ctx.upload(0, q, dim)
        ctx.upload(1, t, dim)
        ctx.set_profiling(True)
        got = ctx.knn(k, 0)
        got_rev = ctx.knn(k, 1)
        st = ctx.stats()
        exact = ctx.knn(k, 0, precision=M.PREC_F32_EXACT)
    exp = orc.knn(_dense(q, dim), _dense(t, dim), k)
    exp_rev = orc.knn(_dense(t, dim), _dense(q, dim), k)
    _same(got, exp)
    _same(exact, exp)
    _same(got_rev, exp_rev)
    if dim <= 2045 and kind not in ("tiny", "huge"):   # the routing: tensor cores up to 2045, nothing beyond
        assert st["candidate_launches"] == 2, (dim, kind)
    elif dim > 2045:
        assert st["candidate_launches"] == 0


@gpu
@pytest.mark.parametrize("dim", [1021, 1960, 2045])
def test_long_operands_and_accumulators(_built, dim):
    """White-box: operand tiles as documented in pack.cu, and raw tcgen05 accumulators of the K-streamed kernel within the
    slop its certificate budgets, ksteps * 2^-21 * (|a| + |b|)^2 + 1e-6 (DESIGN.md §4), on adversarial data: after
    centring every column is +-1 in sign-aligned blocks, so that the partial sums of a row pair grow monotonically."""
    rng = np.random.default_rng(dim)
    nq, nt = 300, 600
    sgn_q = np.where(rng.random((nq, 1)) < 0.5, -1.0, 1.0)
    sgn_t = np.where(rng.random((nt, 1)) < 0.5, -1.0, 1.0)
    src = (sgn_q * np.ones((nq, dim)) * (1 - 2e-3 * rng.random((nq, dim)))).astype(np.float32)
    tgt = (sgn_t * np.ones((nt, dim)) * (1 - 2e-3 * rng.random((nt, dim)))).astype(np.float32)
    ksteps = (dim + 3 + 15) // 16
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        oq, nq16, scale = ctx.debug_operands(0, True)
        ot, nt16, _ = ctx.debug_operands(1, False)
        ot_q, _, _ = ctx.debug_operands(0, False)
        assert oq.shape[1] == (dim + 3 + 63) // 64 * 64 and oq.shape[0] % 256 == 0
        assert np.array_equal(oq[:nq, :dim].astype(np.float32), -2.0 * ot_q[:nq, :dim].astype(np.float32))
        assert np.all(oq[:, dim:dim + 3] == 1) and np.all(oq[:, dim + 3:] == 0) and np.all(ot[:, dim + 3:] == 0)
        x16 = ot_q[:nq, :dim].astype(np.float64)
        np.testing.assert_allclose(nq16[:nq], (x16 ** 2).sum(1), rtol=3e-7)
        assert np.abs(x16).max() <= 1.0
        triple = ot[:nt, dim:dim + 3].astype(np.float64).sum(1)
        np.testing.assert_allclose(triple, (ot[:nt, :dim].astype(np.float64) ** 2).sum(1), rtol=3e-7)
        assert np.all(ot[nt:, dim].astype(np.float64) > 5e4)      # sentinel rows: still far above every valid accumulator
        assert 3 * dim < 6e4
        worst = 0.0
        for (q0, tt) in [(0, 0), (128, 1), (172, 2)]:
            acc = ctx.debug_tc_tile(0, q0, tt)
            a = oq[q0:q0 + 128].astype(np.float64)
            b = ot[tt * 256:(tt + 1) * 256].astype(np.float64)
            exp = a @ b.T
            rows = min(128, nq - q0)
            na = np.sqrt((a[:rows, :dim] ** 2).sum(1) / 4.0)[:, None]
            nb = np.sqrt((b[:, :dim] ** 2).sum(1))[None, :]
            ok = np.abs(exp[:rows]) < 1e4
            err = np.abs(acc[:rows] - exp[:rows])
            budget = (na + nb) ** 2 * (ksteps * 2.0 ** -21) + 1e-6
            assert np.all(err[ok] <= np.broadcast_to(budget, err.shape)[ok])
            worst = max(worst, float((err / np.broadcast_to((na + nb) ** 2 + 1e-30, err.shape))[ok].max()))
        ratio = worst / (ksteps * 2.0 ** -21)
        print("dim %d: max accumulation error / (|a|+|b|)^2 = %.3e, budget %d x 2^-21 = %.3e, margin %.1fx"
              % (dim, worst, ksteps, ksteps * 2.0 ** -21, 1.0 / max(ratio, 1e-30)))
        assert ratio <= 0.25                                      # at least a 4x margin to the measured worst case
        _same(ctx.knn(2, 0), orc.knn(src, tgt, 2))


def _usc(ns, nt, seed=synth.SEED, **kw):
    return synth.make_pair("usc", ns, nt, seed=seed, nan_frac=0.01, **kw)


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "ratio"])
def test_usc_match_equals_oracle(_built, mode):
    src, tgt, dim = _usc(1500, 1800)
    name = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "ratio": M.MODE_RATIO}[mode]
    k = 2
    for prec in (M.PREC_TC_F16, M.PREC_F32_EXACT):
        with M.Context(0) as ctx:
            ctx.upload(0, src, dim)
            ctx.upload(1, tgt, dim)
            got, avg = ctx.match(k, name, 1.1, np.float32(0.9), precision=prec)
        exp, eavg = orc.match(_dense(src, dim), _dense(tgt, dim), k, mode, 1.1, np.float32(0.9))
        assert got.tobytes() == exp.tobytes() and (avg == eavg or (np.isnan(avg) and np.isnan(eavg)))
    assert len(got) > 0


@gpu
@pytest.mark.parametrize("prec", [M.PREC_TC_F16, M.PREC_F32_EXACT], ids=["tc", "exact"])
def test_usc_masked_reverse_pass(_built, monkeypatch, prec):
    """b200m_match's masked reverse pass (compact query operands of the referenced target rows) on USC rows"""
    monkeypatch.setenv("B200M_MASKED_MIN_PAIRS", "0")
    src, tgt, dim = _usc(1200, 1500, seed=3)
    for k in (1, 5):
        with M.Context(0) as ctx:
            ctx.upload(0, src, dim)
            ctx.upload(1, tgt, dim)
            got, avg = ctx.match(k, M.MODE_MUTUAL, 1.1, np.float32(0.9), precision=prec)
        exp, eavg = orc.match(_dense(src, dim), _dense(tgt, dim), k, "mutual", 1.1, np.float32(0.9))
        assert got.tobytes() == exp.tobytes() and avg == eavg


@gpu
def test_usc_overflowed_lists_fall_back_exactly(_built):
    src, tgt, dim = _usc(700, 1100, seed=4)
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        ctx.set_profiling(True)
        got = ctx.knn(5, 0, cand_cap=5)
        st = ctx.stats()
    assert st["candidate_launches"] == 1 and st["rows_flagged"] > 0
    _same(got, orc.knn(_dense(src, dim), _dense(tgt, dim), 5))


@gpu
def test_usc_wide_seam_matcher_classes(_built):
    """ClusterMatcher / LeftToRightMatcher at the wide seam (b200m_match_multiscale), 2 scales, k = 2"""
    import test_gpu_wide_batch as WB
    for mode in ("mutual", "cluster"):
        pr, ts, tt, dim = WB._case("usc", 2, 2, 41, n_sk=700, n_tk=650)
        with M.Context(0) as ctx:
            got, avg = WB._single(ctx, 2, WB.GMODE[mode], pr, dim, ts, tt)
        e, eavg = WB._oracle(mode, 2, pr, ts, tt)
        assert got.tobytes() == e.tobytes() and avg == np.float32(eavg)
        assert len(got) > 0


@gpu
def test_usc_batches(_built):
    """match_wide_batch (= match_many's call), the guessed match_wide_local_batch, knn_batch and match_batch on USC rows"""
    import test_gpu_wide_batch as WB
    import test_gpu_wide_local as WL
    cases = [WB._case("usc", 2, 2, 50 + i, n_sk=500 - 100 * i, n_tk=450) for i in range(3)]
    WB._check("cluster", 2, cases, oracle=True)
    WL._check("mutual", 2, cases, 0.6, [WL._rigid(10 + i, 0.05, 0.05) for i in range(3)])
    pairs = [_usc(300 + 200 * i, 400, seed=60 + i) for i in range(3)]
    pairs = [(s, t) for s, t, _ in pairs]
    with M.Context(0) as ctx:
        kn = ctx.knn_batch(2, pairs, USC_DIM)
        mb = ctx.match_batch(2, M.MODE_MUTUAL, pairs, USC_DIM)
    for (s, t), got, (recs, avg) in zip(pairs, kn, mb):
        _same(got, orc.knn(_dense(s, USC_DIM), _dense(t, USC_DIM), 2))
        e, eavg = orc.match(_dense(s, USC_DIM), _dense(t, USC_DIM), 2, "mutual", M.MATCHING_RATIO_THRESHOLD, M.FLT_MAX)
        assert recs.tobytes() == e.tobytes() and avg == eavg


@gpu
def test_usc_match_many(_built):
    """match_many (one batch call) equals each ClusterMatcher's own match() on USC rows, 2 scales, k = 2"""
    import test_gpu_wide_batch as WB
    makers = []
    for i in range(3):
        pr, ts, tt, dim = WB._case("usc", 2, 2, 70 + i, n_sk=450 + 50 * i, n_tk=400)
        params = M.AlignmentParameters(randomness=2, distance_thr=float(WB.DTHR), cluster_k=40, matching_id=M.MATCHING_CLUSTER)
        makers.append(lambda pr=pr, ts=ts, tt=tt, dim=dim, params=params: M.get_feature_based_matcher_from_parameters(
            [a for a, _ in pr["src_scales"]], [a for a, _ in pr["tgt_scales"]], params, dim=dim, thresholds_src=ts,
            thresholds_tgt=tt, kps_indices_multiscale_src=[m for _, m in pr["src_scales"]],
            kps_indices_multiscale_tgt=[m for _, m in pr["tgt_scales"]], kps_xyz_src=pr["src_kps_xyz"],
            kps_xyz_tgt=pr["tgt_kps_xyz"], iss_radius_src=pr["iss_radius_src"], iss_radius_tgt=pr["iss_radius_tgt"]))
    ref = []
    for mk in makers:
        m = mk()
        ref.append((m.match(), m.get_average_distance()))
    ms = [mk() for mk in makers]
    got = M.match_many(ms)
    for m, g, (r, ravg) in zip(ms, got, ref):
        assert g.tobytes() == r.tobytes() and m.get_average_distance() == ravg
    assert sum(len(g) for g in got) > 0


@gpu
def test_usc_batch_device_equals_host(_built):
    import torch
    from lidar_global_registration_b200 import device as D
    pairs = [_usc(300 + 150 * i, 350, seed=80 + i) for i in range(3)]
    pairs = [(s, t) for s, t, _ in pairs]
    with M.Context(0) as ctx:
        ref = ctx.knn_batch(5, pairs, USC_DIM)
    b = D.GpuBackend(0)
    try:
        dev = [(torch.from_numpy(s).to(b.device), torch.from_numpy(t).to(b.device)) for s, t in pairs]
        got = b.knn_batch(5, dev, USC_DIM)
        torch.cuda.synchronize()
        for (i, d, c), (ri, rd, rc) in zip(got, ref):
            assert np.array_equal(i.cpu().numpy(), ri) and np.array_equal(d.cpu().numpy(), rd) and np.array_equal(c.cpu().numpy(), rc)
    finally:
        b.close()


@gpu
def test_usc_cpp_program_matches_oracle(_built, tmp_path):
    exe = _build_exe()
    ns, nt, k = 400, 500, 2
    src, tgt, dim = _usc(ns, nt, seed=90)
    sp, tp, op = tmp_path / "s.bin", tmp_path / "t.bin", tmp_path / "o.txt"
    src.tofile(sp)
    tgt.tofile(tp)
    r = subprocess.run([exe, str(sp), str(ns), str(tp), str(nt), str(k), str(op)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    s_d, t_d = _dense(src, dim), _dense(tgt, dim)
    exp = {0: orc.knn(s_d, t_d, k), 1: orc.knn(t_d, s_d, k)}
    n_knn, corr, head = 0, [], None
    for line in open(op):
        w = line.split()
        if w[0] == "knn":
            d, i, c = int(w[1]), int(w[2]), int(w[3])
            idx, dist, cnt = exp[d]
            assert c == cnt[i] and [int(x) for x in w[4::2]] == idx[i, :c].tolist()
            assert [np.float32(x) for x in w[5::2]] == dist[i, :c].tolist()
            n_knn += 1
        elif w[0] == "matcher":
            head = (w[2], int(w[3]), np.float32(w[4]))
        elif w[0] == "corr":
            corr.append((int(w[2]), int(w[3]), np.float32(w[4])))
    assert n_knn == ns + nt

    def lattice(n, step):
        i = np.arange(n)
        return np.stack([step * (i % 17), step * ((i // 17) % 13), step * (i // 221)], 1).astype(np.float32)
    sx, tx = lattice(ns, np.float32(0.5)), lattice(nt, np.float32(0.25))
    e, eavg = orc.match_wide("mutual", [(s_d, None)], [(t_d, None)], sx, tx, np.float32(0.3), np.float32(0.2), k, 12,
                             np.float32(np.finfo(np.float32).max))
    assert head == ("LeftToRightMatcher", len(e), np.float32(eavg))
    assert corr == [(int(a), int(b), np.float32(c)) for a, b, c in zip(e["index_query"], e["index_match"], e["distance"])]


@gpu
def test_usc_full_size_routing_and_sampled_rows(_built):
    """20k x 20k USC-1960: the candidate kernel runs (no silent exact path), at most 1 % of the rows overflow, and sampled
    rows equal the oracle"""
    import torch
    s, t, dim = synth.make_pair_torch("usc", 20000, 20000, "cuda:0")
    src, tgt = s.cpu().numpy(), t.cpu().numpy()
    del s, t
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        ctx.set_profiling(True)
        idx, dist, cnt = ctx.knn(1, 0)
        st = ctx.stats()
    print("USC 20k x 20k k=1: candidates %.1f per row, rows flagged %d, candidate kernel %.2f ms, re-rank %.2f ms"
          % (st["candidates"] / 20000, st["rows_flagged"], st["ms_candidates"], st["ms_rerank"]))
    assert st["candidate_launches"] == 1 and st["rows_flagged"] <= 200
    rows = np.random.default_rng(0).choice(20000, 256, replace=False)
    ei, ed, ec = orc.knn(np.ascontiguousarray(src[rows, :dim]), _dense(tgt, dim), 1)
    assert np.array_equal(idx[rows], ei) and np.array_equal(dist[rows], ed) and np.array_equal(cnt[rows], ec)
    torch.cuda.empty_cache()
