"""Descriptor magnitudes over the whole FP32 range, against the oracle byte for byte.

The tensor-core pass is exact only while the certificate's premise holds (DESIGN.md §4): the reference's FP32 distance
`d = pcl::L2_Norm(a, b)` lies within `(1 +- gamma)` of the true distance, up to the subnormal rounding of its terms.
Beyond the upper edge some squared differences or their sum overflow to `inf`; below the lower edge they round to `0`
or to a few subnormal bits.  Either way the reference orders the tied rows by index, which the FP16 geometry cannot
see.  `launch_tc_prepare` routes such data to the exact CUDA-core path.  This file checks:

* the window restated in Python, against float64 and the oracle (CPU);
* a sweep of `2^e`-scaled data across both edges, the +-1e30 limits of earlier builds and subnormal values (GPU);
* far train rows whose distance is `inf`, filters on saturated distances, batches mixing magnitudes (GPU);
* routing through `Context.stats()` one step inside and outside each edge (GPU);
* FP16 operands and accumulators at the smallest and largest in-window scale, and candidates whose distances differ
  below FP16 resolution, answered by the certificate without the fallback (GPU).
"""
import math

import numpy as np
import pytest

from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth
from oracle import oracle as orc

F32 = np.float32
FLT_MAX = float(np.finfo(F32).max)
PRECS = [M.PREC_TC_F16, M.PREC_F32_EXACT]
DIMS = [33, 352, 1960]       # A-resident kernels (kp <= 640) and the K-streamed form (kp > 640)


# ---- the window, restated from launch_tc_prepare (csrc/pack.cu) -------------------------------------------------------
def gamma(dim):
    return (dim + 4) * 2.0 ** -24


def scale_for(maxabs):
    """power of two s with maxabs * s in (0.5, 1], as the float32 ldexpf gives it (inf / 0 beyond float range)"""
    if not (maxabs > 0 and math.isfinite(maxabs)):
        return 1.0
    fr, ex = math.frexp(float(maxabs))
    if fr == 0.5:
        ex -= 1
    if -ex > 127:
        return math.inf
    return float(np.ldexp(F32(1), -ex)) if -ex >= -149 else 0.0


def tc_window(maxabs, dim):
    maxabs = float(F32(maxabs))
    s = scale_for(maxabs)
    if not (math.isfinite(maxabs) and math.isfinite(s) and s > 0):
        return False
    return maxabs == 0 or (dim * 4.0 * maxabs * maxabs * (1 + gamma(dim)) < FLT_MAX and dim * s * s <= 2.0 ** 125)


def upper_edge(dim):
    """largest float32 maxabs inside the window"""
    m = F32(math.sqrt(FLT_MAX / (4.0 * dim * (1 + gamma(dim)))))
    while not tc_window(m, dim):
        m = np.nextafter(m, F32(0))
    while tc_window(np.nextafter(m, F32(np.inf)), dim):
        m = np.nextafter(m, F32(np.inf))
    return float(m)


def lower_edge(dim):
    """smallest float32 maxabs inside the window: just above 2^-(e+1), where s = 2^e is the largest scale allowed"""
    e = int(math.floor((125 - math.log2(dim)) / 2))
    while dim * 4.0 ** e > 2.0 ** 125:
        e -= 1
    return float(np.nextafter(F32(2.0 ** -(e + 1)), F32(np.inf)))


def _outside(edge, hi):
    return float(np.nextafter(F32(edge), F32(np.inf if hi else 0)))


def test_window_edges_are_one_float_apart():
    for dim in (1, 33, 135, 352, 1960, 2045):
        hi, lo = upper_edge(dim), lower_edge(dim)
        assert tc_window(hi, dim) and not tc_window(_outside(hi, True), dim)
        assert tc_window(lo, dim) and not tc_window(_outside(lo, False), dim)
        assert 1e-19 < lo < 1e-17 and 1e17 < hi < 1e19, (dim, lo, hi)   # every descriptor the project knows lives inside
    assert 1.5e18 < upper_edge(33) < 1.7e18
    assert tc_window(0.0, 33) and not tc_window(np.inf, 33) and not tc_window(np.nan, 33)


def _ref_d(a, b):
    """the reference's FP32 distance, one pair at a time (pcl::L2_Norm)"""
    return np.array([orc.l2_norm(np.ascontiguousarray(a[i]), np.ascontiguousarray(b[i])) for i in range(len(a))],
                    np.float64)


def _premise_excess(a, b, s):
    """how far the reference's d^2 leaves [t^2 (1-g)^2, t^2 (1+g)^2] (t = float64 distance), in the scaled units of the
    certificate (s^2 d^2); inf when d is not finite"""
    dim = a.shape[1]
    g = gamma(dim)
    t2 = ((a.astype(np.float64) - b.astype(np.float64)) ** 2).sum(1)
    d = _ref_d(a, b)
    with np.errstate(over="ignore", invalid="ignore"):
        d2 = d * d
        out = np.maximum(d2 - t2 * (1 + g) ** 2, t2 * (1 - g) ** 2 - d2) * s * s
    return np.where(np.isfinite(d), np.maximum(out, 0), np.inf)


def _adversarial_small(dim, unit, rng, n=8):
    """pairs whose every squared difference is subnormal and rounds down by almost half a quantum (2^-150): the
    oracle's d^2 lands almost D 2^-150 below the truth"""
    cands = []
    for x in np.arange(2 ** 14, 2 ** 16, dtype=np.float64) * 2.0 ** -90:     # x^2 in [2^-152, 2^-148]: subnormal
        f = (x * x / 2.0 ** -149) % 1.0
        if 0.45 < f < 0.5:
            cands.append(x)
    cands = np.array(cands)
    a = np.zeros((n, dim), F32)
    b = rng.choice(cands, (n, dim)).astype(F32)
    a[:, 0] = unit              # the spread that sets the scale (equal in both rows: no difference in that column)
    b[:, 0] = unit
    return a, b


@pytest.mark.parametrize("dim", [33, 352, 1960])
def test_window_premise_against_float64(dim):
    """Just inside each edge the reference's FP32 distances obey the certificate's premise: within (1 +- gamma) of the
    float64 distance up to the subnormal term, which stays under the 2^-25 the window budgets (in scaled units, against
    the 1e-6 of slop).  Just outside, some row breaks it: an inf distance above, and the subnormal term at its bound,
    past that budget, below."""
    rng = np.random.default_rng(dim)
    budget = 2.0 ** -25
    # upper edge: rows at +-maxabs in every column, the largest differences the spread allows.  The window keeps a
    # factor (1 + gamma) for the rounding of the sum, so the overflow begins within that factor outside it.
    hi = upper_edge(dim)
    for m, inside in ((hi, True), (float(F32(hi * (1 + gamma(dim)))), False)):
        sign = np.where(rng.random((16, dim)) < 0.5, 1, -1).astype(F32)
        a, b = (sign * F32(m)).astype(F32), (-sign * F32(m)).astype(F32)
        a[1:], b[1:] = a[1:] * F32(0.5), b[1:] * F32(0.25)
        exc = _premise_excess(a, b, scale_for(m))
        if inside:
            assert np.all(exc <= budget), exc.max()
        else:
            assert np.any(np.isinf(exc))
    # lower edge: the bound D 2^-150 s^2 on the subnormal term is within budget at the largest scale the window allows
    # and past it at twice that scale; adversarial rows attain 90 % of the bound at both, so the edge is where the
    # term itself crosses the budget, not a guess
    lo = lower_edge(dim)
    s_in = scale_for(lo)
    a, b = _adversarial_small(dim, F32(lo), rng)
    for s, inside in ((s_in, True), (2 * s_in, False)):
        bound = dim * 2.0 ** -150 * s * s
        assert (bound <= budget) == inside, (s, bound)
        exc = _premise_excess(a, b, s)
        assert np.all(exc <= bound) and exc.max() >= 0.9 * bound, (exc.max(), bound)


@pytest.mark.parametrize("name", sorted(synth.DESCRIPTORS))
def test_generators_are_inside_the_window(name):
    """every synthetic descriptor (and so the benchmark configurations built from them) stays on the tensor cores"""
    src, tgt, dim = synth.make_pair(name, 500, 600, nan_frac=0.01)
    x = np.concatenate([src[:, :dim], tgt[:, :dim]]).astype(np.float64)
    x = x[np.isfinite(x).all(1)]
    maxabs = float(F32(np.abs(x - x.mean(0)).max()))
    assert tc_window(maxabs, dim), (name, maxabs)


# ---- GPU ------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from lidar_global_registration_b200 import build as b200_build
    b200_build.build()
    M.load_library()


def _d(a, dim):
    return np.ascontiguousarray(a[:, :dim])


def _same(got, exp, what=""):
    for x, y in zip(got, exp):
        assert np.array_equal(x, y, equal_nan=True), what


def _check_pair(q, t, dim, ks, what, stats=None):
    """both directions, both precisions, every k: byte for byte the oracle; returns the TC context's stats"""
    exp = {(k, dr): orc.knn(*((_d(q, dim), _d(t, dim)) if dr == 0 else (_d(t, dim), _d(q, dim))), k) for k in ks for dr in (0, 1)}
    out = {}
    for prec in PRECS:
        with M.Context(0) as ctx:
            ctx.upload(0, q, dim)
            ctx.upload(1, t, dim)
            for k in ks:
                for dr in (0, 1):
                    _same(ctx.knn(k, dr, precision=prec), exp[(k, dr)], "%s k=%d dir=%d prec=%d" % (what, k, dr, prec))
            out[prec] = ctx.stats()
    return out[M.PREC_TC_F16]


def _kind(rng, kind, n, dim, e):
    if kind == "uniform":
        a = rng.random((n, dim)) * 2.0 ** e
    elif kind == "clustered":
        protos = rng.random((max(n // 40, 2), dim))
        a = (protos[rng.integers(0, protos.shape[0], n)] + 0.01 * rng.standard_normal((n, dim))) * 2.0 ** e
    else:   # "offset": 2^e +- 2^(e-7): a - b is exact (Sterbenz), the squares and their sum may not be
        a = (1.0 + rng.random((n, dim)) * 2.0 ** -7) * 2.0 ** e
    return a.astype(F32)


def _sweep_exponents(dim):
    hi = math.log2(upper_edge(dim))
    lo = -63 - math.log2(dim) / 2 # differences whose squares reach FLT_MIN (2^-126), summed over D columns
    grid = {0, 100, -100, 99, -99, 101, -101}                         # the +-1e30 limits of earlier builds
    grid |= {int(math.floor(hi)) + d for d in (-2, -1, 0, 1, 2, 3)}  # D (2 maxabs)^2 crosses FLT_MAX
    grid |= {int(lo) + d for d in (-2, 0, 2)}                         # diff^2 crosses FLT_MIN
    grid |= {-75, -73, -71}                                           # ... and the smallest subnormal, 2^-149
    grid |= {int(math.log2(lower_edge(dim))) + d for d in (-1, 0, 1, 2)}
    return sorted(grid)


_SWEEP = [(dim, e) for dim in DIMS for e in _sweep_exponents(dim)]


@gpu
@pytest.mark.parametrize("dim,e", _SWEEP, ids=["d%d_e%d" % c for c in _SWEEP])
def test_magnitude_sweep(lib, dim, e):
    rng = np.random.default_rng(dim * 1000 + e + 500)
    nq, nt = (97, 160) if dim > 640 else (130, 300)
    for kind in ("uniform", "clustered", "offset"):
        both = _kind(rng, kind, nq + nt, dim, e)
        ks = (1, 2, 5, 17) if dim <= 640 else (1, 5, 17)
        _check_pair(both[:nq], both[nq:], dim, ks, "%s dim=%d e=%d" % (kind, dim, e))


@gpu
@pytest.mark.parametrize("dim", DIMS)
def test_subnormal_values(lib, dim):
    """values that are FP32 subnormals themselves: the exact path answers, bit for bit"""
    rng = np.random.default_rng(dim + 7)
    for e in (-130, -140, -148):
        both = (rng.random((200, dim)) * 2.0 ** e).astype(F32)
        assert np.any((both != 0) & (np.abs(both) < np.finfo(F32).tiny))
        st = _check_pair(both[:80], both[80:], dim, (1, 2, 5), "subnormal dim=%d e=%d" % (dim, e))
        assert st["candidate_launches"] == 0


@gpu
@pytest.mark.parametrize("dim", [33, 352])
def test_far_rows_come_last_by_index(lib, dim):
    """train rows that are finite but so far away that their distance is inf: last, ordered by index, also when k
    exceeds the rows at a finite distance"""
    rng = np.random.default_rng(dim)
    q = rng.random((50, dim)).astype(F32)
    t = rng.random((9, dim)).astype(F32)
    t[[2, 5, 6], 0] = F32(1e20)
    t[5, 1] = F32(-1e20)
    for k in (1, 5, 6, 7, 9):
        _check_pair(q, t, dim, (k,), "far rows dim=%d" % dim)
    idx, dist, cnt = orc.knn(q, t, 9)
    assert np.all(cnt == 9) and np.all(idx[:, 6:] == [2, 5, 6]) and np.all(np.isinf(dist[:, 6:]))
    # one far row among many ordinary ones, and one column at 1e18 with the rest at unit scale
    t2 = rng.random((700, dim)).astype(F32)
    t2[333, dim // 2] = F32(1e20)
    _check_pair(q, t2, dim, (1, 2, 5, 17), "one far row dim=%d" % dim)
    t3 = rng.random((700, dim)).astype(F32)
    q3 = q.copy()
    t3[:, 3] *= F32(1e18)
    q3[:, 3] *= F32(1e18)
    _check_pair(q3, t3, dim, (1, 2, 5), "one column at 1e18, dim=%d" % dim)


_MODES = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "ratio": M.MODE_RATIO}


def _match_same(ctx, q, t, dim, k, mode, thr, prec, what):
    got, avg = ctx.match(k, _MODES[mode], 1.1, thr, precision=prec)
    exp, eavg = orc.match(_d(q, dim), _d(t, dim), k, mode, 1.1, thr)
    assert got.tobytes() == exp.tobytes(), what
    assert avg == eavg or (np.isnan(avg) and np.isnan(eavg)), (what, avg, eavg)
    return exp, eavg


@gpu
@pytest.mark.parametrize("dim", [33, 1960])
def test_filters_on_saturated_distances(lib, dim):
    """one-sided, mutual and ratio (inf >= 1.1f * inf) on distances that are all inf or all 0, with and without a
    distance threshold; the average distance inf, 0, and that of a call without a valid query"""
    rng = np.random.default_rng(dim + 3)
    cases = {"inf": (rng.random((120, dim)) * 2.0 ** 70).astype(F32),
             "zero": (rng.random((120, dim)) * 2.0 ** -90).astype(F32),
             "mixed": np.concatenate([rng.random((60, dim)), rng.random((60, dim)) * 1e20]).astype(F32)}
    nan_q = rng.random((30, dim)).astype(F32)
    nan_q[:, 0] = np.nan
    seen = set()
    for name, both in cases.items():
        q, t = both[:50], both[50:]
        for prec in PRECS:
            with M.Context(0) as ctx:
                ctx.upload(0, q, dim)
                ctx.upload(1, t, dim)
                for mode in _MODES:
                    for k in (2, 5):
                        for thr in (F32(FLT_MAX), F32(0.5), F32(0.0)):
                            _, eavg = _match_same(ctx, q, t, dim, k, mode, thr, prec, (name, mode, k, thr, prec))
                            seen.add("inf" if np.isinf(eavg) else "zero" if eavg == 0 else "finite")
        with M.Context(0) as ctx:
            ctx.upload(0, nan_q, dim)
            ctx.upload(1, t, dim)
            for mode in _MODES:
                _match_same(ctx, nan_q, t, dim, 2, mode, F32(FLT_MAX), M.PREC_TC_F16, (name, "no valid query", mode))
    assert {"inf", "zero"} <= seen, seen


def _batch_sets(dim, rng):
    """pairs at 1e-3, 1, an offset of 1e4, 1e20 and 1e-25"""
    out = []
    for i, (scale, off) in enumerate(((1e-3, 0), (1, 0), (1, 1e4), (1e20, 0), (1e-25, 0))):
        ns, nt = 90 + 13 * i, 140 - 11 * i
        out.append(((rng.random((ns, dim)) * scale + off).astype(F32), (rng.random((nt, dim)) * scale + off).astype(F32)))
    return out


@gpu
@pytest.mark.parametrize("dim", [33, 1960])
def test_batches_mixing_magnitudes(lib, dim):
    """one pair at 1e20 sends the whole batch to the exact path; every pair still equals its single-pair call and the
    oracle, host and device forms alike"""
    rng = np.random.default_rng(dim + 11)
    pairs = _batch_sets(dim, rng)
    k = 2
    with M.Context(0) as ctx:
        got = ctx.knn_batch(k, pairs, dim)
        st = ctx.stats()
        mgot = {mode: ctx.match_batch(k, _MODES[mode], pairs, dim, 1.1, F32(0.5)) for mode in _MODES}
    assert st["candidate_launches"] == 0
    for p, (s, t) in enumerate(pairs):
        _same(got[p], orc.knn(s, t, k), "knn_batch pair %d" % p)
        with M.Context(0) as ctx:
            ctx.upload(0, s, dim)
            ctx.upload(1, t, dim)
            _same(ctx.knn(k, 0), got[p], "single pair %d" % p)
            for mode in _MODES:
                one, oavg = ctx.match(k, _MODES[mode], 1.1, F32(0.5))
                recs, avg = mgot[mode][p]
                assert recs.tobytes() == one.tobytes() and (avg == oavg or (np.isnan(avg) and np.isnan(oavg))), (mode, p)
                exp, eavg = orc.match(s, t, k, mode, 1.1, F32(0.5))
                assert recs.tobytes() == exp.tobytes(), (mode, p)
    # the batch without its out-of-window pairs runs the candidate kernel
    with M.Context(0) as ctx:
        ctx.knn_batch(k, pairs[:3], dim)
        assert ctx.stats()["candidate_launches"] > 0
    # matcher classes at the wide seam, one scale per pair
    xrng = np.random.default_rng(5)
    wide = []
    for s, t in pairs:
        sx = np.zeros((len(s), 4), F32)
        tx = np.zeros((len(t), 4), F32)
        sx[:, :3] = xrng.random((len(s), 3)) * 4
        tx[:, :3] = xrng.random((len(t), 3)) * 4
        wide.append(dict(src_scales=[(s, None)], tgt_scales=[(t, None)], src_kps_xyz=sx, tgt_kps_xyz=tx,
                         iss_radius_src=F32(0.05), iss_radius_tgt=F32(0.05)))
    dthr = F32(0.7)
    for mode in ("one_sided", "mutual"):
        gm = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL}[mode]
        with M.Context(0) as ctx:
            wgot = ctx.match_wide_batch(k, gm, wide, dim, 40, dthr)
            for p, pr in enumerate(wide):
                one = ctx.match_wide(k, gm, pr["src_scales"], pr["tgt_scales"], pr["src_kps_xyz"], pr["tgt_kps_xyz"],
                                     pr["iss_radius_src"], pr["iss_radius_tgt"], dim, 40, dthr)
                exp, eavg = orc.match_wide(mode, pr["src_scales"], pr["tgt_scales"], pr["src_kps_xyz"][:, :3],
                                           pr["tgt_kps_xyz"][:, :3], pr["iss_radius_src"], pr["iss_radius_tgt"], k, 40, dthr)
                assert wgot[p][0].tobytes() == one[0].tobytes(), (mode, p)
                assert one[0].tobytes() == exp.tobytes(), (mode, p)
                assert wgot[p][1] == one[1] and (one[1] == eavg or (np.isnan(one[1]) and np.isnan(eavg))), (mode, p)
        local = [dict(pr, src_kps_moved=pr["src_kps_xyz"], tgt_kps_moved=pr["tgt_kps_xyz"]) for pr in wide]
        with M.Context(0) as ctx:
            lgot = ctx.match_wide_local_batch(k, gm, local, 0.5, dim)
            for p, pr in enumerate(local):
                lone = ctx.match_wide_local_batch(k, gm, [pr], 0.5, dim)[0]
                assert lgot[p][0].tobytes() == lone[0].tobytes(), (mode, p)
                assert lgot[p][1] == lone[1] or (np.isnan(lgot[p][1]) and np.isnan(lone[1])), (mode, p)
    # device-resident forms equal the host forms
    torch = pytest.importorskip("torch")
    from lidar_global_registration_b200 import device as D
    be = D.GpuBackend(0)
    tp = [(torch.from_numpy(s).cuda(), torch.from_numpy(t).cuda()) for s, t in pairs]
    dgot = be.knn_batch(k, tp, dim)
    for p in range(len(pairs)):
        _same([x.cpu().numpy() for x in dgot[p]], got[p], "knn_batch_device pair %d" % p)
    for mode in _MODES:
        dm = be.match_batch(k, _MODES[mode], tp, dim, 1.1, F32(0.5))
        for p in range(len(pairs)):
            recs = dm[p][0].cpu().numpy()
            assert recs.tobytes() == mgot[mode][p][0].tobytes(), (mode, p)
    twide = [dict(pr, src_scales=[(torch.from_numpy(pr["src_scales"][0][0]).cuda(), None)],
                  tgt_scales=[(torch.from_numpy(pr["tgt_scales"][0][0]).cuda(), None)],
                  src_kps_xyz=torch.from_numpy(pr["src_kps_xyz"]).cuda(), tgt_kps_xyz=torch.from_numpy(pr["tgt_kps_xyz"]).cuda())
             for pr in wide]
    with M.Context(0) as ctx:
        href = ctx.match_wide_batch(k, M.MODE_MUTUAL, wide, dim)
    dw = be.match_wide_batch(k, M.MODE_MUTUAL, twide, dim)
    for p in range(len(pairs)):
        assert dw[p][0].cpu().numpy().tobytes() == href[p][0].tobytes(), p
    tlocal = [dict(pr, src_kps_moved=pr["src_kps_xyz"], tgt_kps_moved=pr["tgt_kps_xyz"]) for pr in twide]
    with M.Context(0) as ctx:
        lref = ctx.match_wide_local_batch(k, M.MODE_MUTUAL, local, 0.5, dim)
    dl = be.match_wide_local_batch(k, M.MODE_MUTUAL, tlocal, 0.5, dim)
    for p in range(len(pairs)):
        assert dl[p][0].cpu().numpy().tobytes() == lref[p][0].tobytes(), p


def _symmetric(rng, n, dim, edge, unit):
    """source X and target -X (permuted): the common centre is exactly 0 and the centred spread exactly `edge`.
    Columns alternate between a coarse grid of +-unit and a fine one below 2^-14 unit (FP16 subnormals once scaled),
    so every partial sum the statistics pass forms is exact."""
    x = np.zeros((n, dim), np.float64)
    coarse = np.arange(dim) % 3 != 2
    x[:, coarse] = rng.integers(-256, 257, (n, int(coarse.sum()))) / 256.0
    x[:, ~coarse] = rng.integers(-1023, 1024, (n, int((~coarse).sum()))) * 2.0 ** -24
    src = (x * unit).astype(F32)
    src[0, 0] = F32(edge)
    tgt = -src[rng.permutation(n)]
    assert np.abs(np.concatenate([src, tgt])).max() == F32(edge)
    return src, tgt


def _edge_cases(dim):
    hi, lo = upper_edge(dim), lower_edge(dim)
    return [("hi_in", hi, True), ("hi_out", _outside(hi, True), False), ("lo_in", lo, True), ("lo_out", _outside(lo, False), False)]


def _unit(edge):
    return 2.0 ** (math.frexp(edge)[1] - 2)    # a power of two below the edge


@gpu
@pytest.mark.parametrize("dim", DIMS)
def test_routing_at_the_edges(lib, dim):
    """one float inside each edge the candidate kernel runs, one float outside it does not; both answer as the oracle"""
    rng = np.random.default_rng(dim + 1)
    for name, edge, inside in _edge_cases(dim):
        assert tc_window(edge, dim) == inside
        src, tgt = _symmetric(rng, 300, dim, edge, _unit(edge))
        st = _check_pair(src, tgt, dim, (1, 2), "%s dim=%d" % (name, dim))
        assert (st["candidate_launches"] > 0) == inside, (name, st)


@gpu
@pytest.mark.parametrize("name", sorted(synth.DESCRIPTORS))
def test_routing_of_the_generators(lib, name):
    """the synthetic descriptors, and the benchmark configurations built from them, run the candidate kernel and need
    no fallback beyond the usual overflowed rows"""
    src, tgt, dim = synth.make_pair(name, 2000, 2100, nan_frac=0.01)
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        got = ctx.knn(2, 0)
        st = ctx.stats()
    assert st["candidate_launches"] > 0 and st["rows_flagged"] < st["rows_total"] // 10, st
    _same(got, orc.knn(_d(src, dim), _d(tgt, dim), 2))


def _ks_budget(dim):
    kp = -(-(dim + 3) // 64) * 64
    return ((dim + 3 + 15) // 16) * 2.0 ** -21 if kp > 640 else 2.0 ** -16


@gpu
@pytest.mark.parametrize("dim", DIMS)
@pytest.mark.parametrize("edge", ["lo", "hi"])
def test_operands_and_accumulators_at_the_edges(lib, dim, edge):
    """FP16 operands = numpy's round-to-nearest of (x - 0) * s, subnormals included; |dx| within DESIGN §4's bound
    against float64; raw accumulators within slop"""
    rng = np.random.default_rng(dim + (0 if edge == "lo" else 1))
    m = lower_edge(dim) if edge == "lo" else upper_edge(dim)
    s_exp = scale_for(m)
    unit = 2.0 ** -math.log2(s_exp) if edge == "lo" else _unit(m)   # lo: 1/s, the smallest power of two with this scale
    src, tgt = _symmetric(rng, 260, dim, unit if edge == "lo" else m, unit)
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        oq, _, scale = ctx.debug_operands(0, True)
        ot_q, _, _ = ctx.debug_operands(0, False)
        ot, _, _ = ctx.debug_operands(1, False)
        assert scale == s_exp
        x16 = (src.astype(np.float64) * scale).astype(F32).astype(np.float16)
        assert ot_q[:len(src), :dim].tobytes() == x16.tobytes()
        assert np.any((x16 != 0) & (np.abs(x16) < np.finfo(np.float16).tiny)), "no FP16 subnormal operand"
        assert np.array_equal(oq[:len(src), :dim].astype(np.float64), -2.0 * x16.astype(np.float64))
        x = src.astype(np.float64) * scale
        dx = np.sqrt(((x16.astype(np.float64) - x) ** 2).sum(1))
        bound = 2.0 ** -11 * (1 + 2.0 ** -9) * np.sqrt((x16.astype(np.float64) ** 2).sum(1)) + 2.0 ** -24 * math.sqrt(dim)
        assert np.all(dx <= bound)
        for q0, tt in ((0, 0), (128, 1)):
            acc = ctx.debug_tc_tile(0, q0, tt)
            a = oq[q0:q0 + 128].astype(np.float64)
            b = ot[tt * 256:(tt + 1) * 256].astype(np.float64)
            exp = a @ b.T
            rows = min(128, len(src) - q0)
            na = np.sqrt((a[:rows, :dim] ** 2).sum(1) / 4.0)[:, None]
            nb = np.sqrt((b[:, :dim] ** 2).sum(1))[None, :]
            ok = np.abs(exp[:rows]) < 1e4
            err = np.abs(acc[:rows] - exp[:rows])
            budget = np.broadcast_to((na + nb) ** 2 * _ks_budget(dim) + 1e-6, err.shape)
            assert np.all(err[ok] <= budget[ok])


def _margin_case(dim, rng, n_q=256, m=6, r=0.05):
    """per query m train rows at distance r (1 + eps), eps spread over [2^-22, 2^-12] (finer than FP16 resolution,
    coarser than FP32), every other row far away"""
    q = (rng.random((n_q, dim)) * 2 - 1).astype(F32)
    near = []
    for i in range(n_q):
        u = rng.standard_normal((m, dim))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        eps = 2.0 ** rng.uniform(-22, -12, m)
        near.append(q[i].astype(np.float64) + r * (1 + eps)[:, None] * u)
    far = rng.random((300, dim)) * 2 - 1
    t = np.concatenate(near + [far]).astype(F32)
    return q, t[rng.permutation(len(t))]


MARGIN_VARIANTS = [("default", {}), ("splits2", {"B200M_TC_SPLITS": "2"}), ("splits4", {"B200M_TC_SPLITS": "4"}),
                   ("alt1", {"B200M_TC_ALT": "1"}), ("alt2", {"B200M_TC_ALT": "2"})]


@gpu
@pytest.mark.parametrize("variant", [v[0] for v in MARGIN_VARIANTS])
@pytest.mark.parametrize("dim", DIMS)
def test_certificate_at_its_margin(lib, monkeypatch, dim, variant):
    """the certificate, not the fallback, answers rows whose nearest neighbours are tied at FP16 resolution"""
    for name, val in dict(MARGIN_VARIANTS)[variant].items():
        monkeypatch.setenv(name, val)
    rng = np.random.default_rng(dim + 17)
    q, t = _margin_case(dim, rng)
    with M.Context(0) as ctx:
        ctx.upload(0, q, dim)
        ctx.upload(1, t, dim)
        for k in (1, 2, 5):
            ctx.reset_stats()
            got = ctx.knn(k, 0)
            st = ctx.stats()
            assert st["candidate_launches"] > 0 and st["rows_flagged"] == 0, (k, st)
            _same(got, orc.knn(q, t, k), "margin dim=%d k=%d %s" % (dim, k, variant))
