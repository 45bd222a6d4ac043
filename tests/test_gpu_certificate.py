"""The candidate certificate (DESIGN.md §4), checked against a float64 restatement of it.

The tensor-core pass is bit-exact only because `thr(T)` over-approximates the accumulator of every exact top-k member.
A threshold that is too tight drops a neighbour silently: the re-rank never sees it and no row is flagged.  This file
states the bound twice in float64 -- `thr_design` (DESIGN §4 as written, no guards) and `thr_kernel` (the kernel's own
padded constants) -- and checks it four ways:

a. white box (GPU): the lists and per-list thresholds of the last candidate launch (`Context.debug_candidate_lists`)
   against every raw accumulator (`debug_tc_tile`): recorded values bit for bit, every threshold >= thr_design(T_true),
   the single-list threshold pinned to thr_kernel of the list's own k-th smallest, and every column under
   thr_design(T_true) in the lists -- for every kernel family (chosen through D) and epilogue variant;
b. a sensitivity self-check inside each case: for each term of the certificate, rows whose threshold would fall below
   thr_design(T_true) without it (so the case can see that term);
c. black box: FP16 images rounded adversarially on a dyadic grid push every query's true neighbours behind exact rivals;
   byte-for-byte parity with the oracle through every entry point, and a float64 proof that eta = 0 would lose them;
d. the A-resident kernels' accumulators on sign-aligned rows within a quarter of their slop.
"""
import math

import numpy as np
import pytest

from lidar_global_registration_b200 import matcher as M
from oracle import oracle as orc

gpu = pytest.mark.gpu
F32 = np.float32
U11 = 2.0 ** -11 * (1 + 2.0 ** -9)      # FP16 round-to-nearest, relative, incl. the FP32 rounding of (x - c) * s


def ksteps_of(dim):
    return (dim + 3 + 15) // 16


def k_streamed(dim):
    return -(-(dim + 3) // 64) * 64 > 640


def gamma(dim):
    return (dim + 4) * 2.0 ** -24


def _slop(ab, dim, drop=None):
    if k_streamed(dim):
        per = 2.0 ** -16 if drop == "ks_slop" else ksteps_of(dim) * 2.0 ** -21
    else:
        per = 0.0 if drop == "slop" else 2.0 ** -16
    return ab * ab * per + 1e-6


def thr_design(T, na, bmax, dim):
    """DESIGN §4: ((sqrt(T + na + slop) + eta)(1 + g)/(1 - g) + eta)^2 - na + slop, eta = |da| + |db| bounds summed"""
    T, na = np.asarray(T, np.float64), np.asarray(na, np.float64)
    ab = np.sqrt(na) + bmax
    eta = U11 * ab + 2 * 2.0 ** -24 * math.sqrt(dim)
    g = gamma(dim)
    slop = _slop(ab, dim)
    with np.errstate(invalid="ignore"):
        R = (np.sqrt(np.maximum(T + na + slop, 0)) + eta) * (1 + g) / (1 - g) + eta
    return np.where(np.isfinite(T), R * R - na + slop, np.inf)


def thr_kernel(T, na, bmax, dim, drop=None):
    """cand_threshold with the constants the kernel stores per row (candidates_tc.cu), in float64; `drop` removes one
    term as a weakened certificate would: eta, gfac, slop, ks_slop, bmax (ab = |a16|)"""
    T, na = np.asarray(T, np.float64), np.asarray(na, np.float64)
    ab = np.sqrt(na) + (0.0 if drop == "bmax" else bmax)
    eta = 0.0 if drop == "eta" else ab * 2.0 ** -11 * (1 + 2.0 ** -9) + 2.0 ** -22 * math.sqrt(dim)
    slop = _slop(ab, dim, drop)
    gfac = 1.0 if drop == "gfac" else 1 + 2.2 * (dim + 4) * 2.0 ** -24
    with np.errstate(invalid="ignore"):
        R = (np.sqrt(np.maximum(T + na + slop, 0)) * (1 + 2.0 ** -20) + eta) * gfac + eta
    R2 = R * R
    return np.where(np.isfinite(T), (R2 - na) + slop + 2.0 ** -20 * (R2 + na), np.inf)


def fp32_slack(thr, na):
    """how far the kernel's FP32 evaluation of cand_threshold may sit from thr_kernel in float64 (the size of its guards)"""
    return 2.0 ** -20 * (np.abs(thr) + 2 * np.asarray(na, np.float64)) + 2.0 ** -20


def invert_kernel(thr, na, bmax, dim):
    """the T at which thr_kernel reaches `thr` (bisection; thr_kernel is monotone): the k-th smallest a list ended with"""
    thr = np.asarray(thr, np.float64)
    na = np.broadcast_to(np.asarray(na, np.float64), thr.shape)
    lo = np.minimum(thr, 0) - na - 1.0
    hi = np.where(np.isfinite(thr), thr, 0.0)
    for _ in range(80):
        mid = 0.5 * (lo + hi)
        up = thr_kernel(mid, na, bmax, dim) > thr
        hi, lo = np.where(up, mid, hi), np.where(up, lo, mid)
    return np.where(np.isfinite(thr), lo, np.inf)


TERMS_ARES = ["eta", "gfac", "slop", "bmax"]
TERMS_KS = ["eta", "gfac", "ks_slop", "bmax"]


# ---- CPU: the two restatements -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [33, 61, 125, 352, 637, 638, 1960])
def test_kernel_constants_cover_the_design(dim):
    """the kernel's padded constants never fall below DESIGN §4's bound, and every weakened term does somewhere"""
    rng = np.random.default_rng(dim)
    na = np.concatenate([[0.0], 10.0 ** rng.uniform(-6, math.log10(dim), 4000)])
    bmax = math.sqrt(dim) * 0.9
    T = np.concatenate([-na[:2000] + 10.0 ** rng.uniform(-8, 1, 2000), rng.uniform(-1, 1, 2001) * dim])
    T = np.maximum(T, -na)
    assert np.all(thr_kernel(T, na, bmax, dim) >= thr_design(T, na, bmax, dim))
    for term in (TERMS_KS if k_streamed(dim) else TERMS_ARES):
        assert np.any(thr_kernel(T, na, bmax, dim, term) < thr_design(T, na, bmax, dim)), term
    t_back = invert_kernel(thr_kernel(T, na, bmax, dim), na, bmax, dim)
    np.testing.assert_allclose(t_back, T, rtol=1e-9, atol=1e-9 * dim)


# ---- a / b: white box, every kernel family --------------------------------------------------------------------------------
def _band_case(dim, regime, rng, n_q=200, m=8, n_far=6300):
    """per query m train rows at distance r (1 + eps), eps log-uniform over [2^-24, 2^-3]; far rows elsewhere; a few NaN
    rows on both sides.  centre: queries at the centre of the data (|a16| ~ 0); far: queries far from it with close
    neighbours (|a16|^2 >> d^2)."""
    far = rng.uniform(-1, 1, (n_far, dim))
    if regime == "centre":
        # |a|^2 under a tenth of bmax^2, queries 0.2 sqrt(D) apart; r large enough that the gfac term (~ gamma d^2)
        # outgrows the kernel's padding of eta (~ 2^-22 sqrt(D) d)
        q = rng.normal(0, 0.15, (n_q, dim))
        r = max(0.05 * math.sqrt(dim), 8.0 / math.sqrt(dim))
    else:
        q = np.sign(rng.standard_normal((n_q, dim))) * rng.uniform(0.6, 0.9, (n_q, dim))
        r = 2e-3 * math.sqrt(dim)
    band = []
    for i in range(n_q):
        u = rng.standard_normal((m, dim))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        eps = 2.0 ** rng.uniform(-24, -3, m)
        band.append(q[i] + r * (1 + eps)[:, None] * u)
    t = np.concatenate(band + [far])[rng.permutation(n_q * m + n_far)].astype(F32)
    q = q.astype(F32)
    q[rng.choice(n_q, 3, replace=False)] = np.nan
    t[rng.choice(len(t), 5, replace=False)] = np.nan
    return q, t


def _accumulators(ctx, nq, nt):
    """every raw accumulator of direction 0: [nq][n_pad] (query rows of one launch, train rows in side order)"""
    n_pad = -(-nt // 256) * 256
    acc = np.empty((nq, n_pad), np.float32)
    for q0 in range(0, nq, 128):
        rows = min(128, nq - q0)
        for tt in range(n_pad // 256):
            acc[q0:q0 + rows, tt * 256:(tt + 1) * 256] = ctx.debug_tc_tile(0, q0, tt)[:rows]
    return acc


def _t_emulated(acc_row_list, k):
    """the k-th smallest a one-list EH = 1 thread ends with: its first 128 columns one by one, then 32-column chunk minima"""
    first = acc_row_list[:, :128]
    rest = acc_row_list[:, 128:].reshape(len(acc_row_list), -1, 32).min(axis=2)
    return np.sort(np.concatenate([first, rest], axis=1).astype(np.float64), axis=1)[:, k - 1]


def check_lists(lists, acc, valid_q, valid_t, na, bmax, dim, k, what, sweep=None, bmax_kernel=None):
    """assertions a. on one launch's lists; returns {term: rows whose threshold would fall below thr_design without it}.
    bmax: the bound of the columns these rows may see (thr_design); bmax_kernel: the one the launch uses (batch-wide);
    sweep: the (first, end) train rows the rows' launch sweeps (a batch pair's own), default all"""
    bk = bmax if bmax_kernel is None else bmax_kernel
    kind, cap, cnt, idx, val, thr = (lists[x] for x in ("kind", "cap", "cnt", "idx", "val", "thr"))
    n_lists, n_rows = cnt.shape
    assert n_rows == len(acc), what
    assert np.all(cnt[:, valid_q] <= cap), (what, "overflowed list")
    masked = np.where(valid_t[None, :], acc[:, :len(valid_t)].astype(np.float64), np.inf)
    T_true = np.sort(masked, axis=1)[:, k - 1]
    design = thr_design(T_true, na, bmax, dim)
    rows = np.nonzero(valid_q)[0]
    terms = TERMS_KS if k_streamed(dim) else TERMS_ARES
    sens = {t: 0 for t in terms}
    for r in rows:
        need = np.nonzero(masked[r] < design[r])[0]          # every column a correct list must hold
        have = set()
        for l in range(n_lists):
            c = min(int(cnt[l, r]), cap)
            ent = idx[l, r, :c]
            if kind == 2:
                have.update((ent // 32).tolist())
                lo = ent[:, None] + np.arange(32)[None, :]
                assert np.array_equal(val[l, r, :c], acc[r][lo].min(axis=1)), (what, "chunk minimum", r, l)
                assert np.all(ent % 32 == 0), (what, r, l)
            else:
                have.update(ent.tolist())
                if kind == 1:
                    assert val[l, r, :c].tobytes() == acc[r, ent].tobytes(), (what, "recorded value", r, l)
        key = need // 32 if kind == 2 else need
        missing = [int(j) for j, kk in zip(need, key) if int(kk) not in have]
        assert not missing, (what, "row %d misses columns %s under thr_design(T_true)" % (r, missing[:8]))
        if kind:
            assert np.all(thr[:, r].astype(np.float64) >= design[r]), (what, "threshold below thr_design", r, thr[:, r],
                                                                       design[r], T_true[r])
    if kind:
        t_fin = invert_kernel(thr[:, rows].astype(np.float64), na[rows][None, :], bk, dim)
        for term in terms:
            # (the FP32 evaluation of the mutant's formula errs by about one sqrt.approx: 2^-21 of R^2)
            mut = thr_kernel(t_fin, na[rows][None, :], bk, dim, term) + 2.0 ** -21 * (np.abs(thr[:, rows]) + 2 * na[rows][None, :])
            sens[term] = int(np.any(mut < design[rows][None, :], axis=0).sum())
        if kind == 1 and n_lists == 1:     # one list: its final k-th smallest is known exactly -> pin the threshold
            lo, hi = sweep if sweep is not None else (0, acc.shape[1])
            t_em = _t_emulated(acc[rows][:, lo:hi], k)
            pin = thr_kernel(t_em, na[rows], bk, dim)
            got = thr[0, rows].astype(np.float64)
            slack = fp32_slack(pin, na[rows])
            bad = np.nonzero(np.abs(got - pin) > slack)[0]
            assert len(bad) == 0, (what, "threshold off thr_kernel(T_final)", rows[bad[:4]], got[bad[:4]], pin[bad[:4]])
    return kind, n_lists, sens


FAMILIES = [33, 61, 62, 125, 126, 352, 637, 638, 1960]
VARIANTS = {"default": {}, "splits1": {"B200M_TC_SPLITS": "1"}, "splits4": {"B200M_TC_SPLITS": "4"},
            "alt0": {"B200M_TC_ALT": "0"}, "alt1": {"B200M_TC_ALT": "1"}, "alt2": {"B200M_TC_ALT": "2"},
            "alt4": {"B200M_TC_ALT": "4"}, "alt5": {"B200M_TC_ALT": "5"}, "mcast": {"B200M_TC_MODE": "mcast"}}


def _cases():
    out = []
    for dim in FAMILIES:
        for v in VARIANTS:
            if v.startswith("alt") and dim > 61:
                continue              # the epilogue layouts exist for one-atom descriptors only
            if v == "mcast" and dim > 509:
                continue              # K-streamed: CTA-pair mode only; D = 637: no two-stage ring fits beside the query tile
            out.append((dim, v))
    return out


@gpu
@pytest.mark.parametrize("dim,variant", _cases())
def test_thresholds_against_the_restatement(monkeypatch, dim, variant):
    for name, val in VARIANTS[variant].items():
        monkeypatch.setenv(name, val)
    rng = np.random.default_rng(1000 + dim)
    seen = {}
    for regime in ("centre", "far"):
        q, t = _band_case(dim, regime, rng)
        valid_q, valid_t = ~np.isnan(q).any(1), ~np.isnan(t).any(1)
        with M.Context(0) as ctx:
            ctx.upload(0, q, dim)
            ctx.upload(1, t, dim)
            got = {}
            for k in (1, 2, 5):
                ctx.reset_stats()
                got[k] = (ctx.knn(k, 0, cand_cap=512), ctx.debug_candidate_lists(), ctx.stats())
            _, na, _ = ctx.debug_operands(0, True)
            ot, nt16, _ = ctx.debug_operands(1, False)
            acc = _accumulators(ctx, len(q), len(t))
        bmax = float(np.sqrt((ot[:len(t)][valid_t, :dim].astype(np.float64) ** 2).sum(1)).max())
        na = na[:len(q)].astype(np.float64)
        for k in (1, 2, 5):
            res, lists, st = got[k]
            what = "dim=%d %s %s k=%d" % (dim, variant, regime, k)
            assert st["candidate_launches"] == 1 and st["rows_flagged"] == 0, (what, st)
            _same(res, orc.knn(q, t, k), what)
            kind, n_lists, sens = check_lists(lists, acc, valid_q, valid_t, na, bmax, dim, k, what)
            for term, n in sens.items():
                seen[term] = seen.get(term, 0) + n
            print("%s: kind %d, %d lists, rows the case sees per term: %s" % (what, kind, n_lists, sens))
    if kind:
        blind = [term for term, n in seen.items() if n == 0]
        assert not blind, ("dim=%d %s: no row would see these terms removed" % (dim, variant), blind)


def _same(got, exp, what=""):
    for a, b, name in zip(got, exp, ("idx", "dist", "cnt")):
        assert np.array_equal(a, b), "%s: %s differs from the oracle" % (what, name)


@gpu
@pytest.mark.parametrize("dim", [61, 352])
def test_batch_thresholds_use_the_batch_bound(dim):
    """knn_batch (the SEG kernels): pairs of very different norms; each pair's rows are held to thr_design with their own
    pair's bound, and the lists stay inside their own pair"""
    rng = np.random.default_rng(dim + 5)
    pairs = []
    for scale_ in (1.0, 0.125, 0.5):
        q, t = _band_case(dim, "centre", rng, n_q=100, m=8, n_far=700)
        pairs.append(((q * scale_).astype(F32), (t * scale_).astype(F32)))
    with M.Context(0) as ctx:
        for k in (1, 2, 5):
            ctx.reset_stats()
            res = ctx.knn_batch(k, pairs, dim, cand_cap=512)
            st = ctx.stats()
            lists = ctx.debug_candidate_lists()
            assert st["rows_flagged"] == 0, st
            for p, (q, t) in enumerate(pairs):
                _same(res[p], orc.knn(q, t, k), "batch dim=%d pair %d k=%d" % (dim, p, k))
        # the batch's sides: each set padded to 256 rows, in pair order
        _, na, scale = ctx.debug_operands(0, True)
        ot, _, _ = ctx.debug_operands(1, False)
        qs = [-(-len(q) // 256) * 256 for q, _ in pairs]
        ts = [-(-len(t) // 256) * 256 for _, t in pairs]
        nq_all, nt_all = sum(qs), sum(ts)
        acc = _accumulators(ctx, nq_all, nt_all)
    valid_all = np.zeros(nt_all, bool)
    t0 = 0
    for p, (_, t) in enumerate(pairs):
        valid_all[t0:t0 + len(t)] = ~np.isnan(t).any(1)
        t0 += ts[p]
    bmax_batch = float(np.sqrt((ot[:nt_all][valid_all, :dim].astype(np.float64) ** 2).sum(1)).max())
    q0 = t0 = 0
    for p, (q, t) in enumerate(pairs):
        valid_q = np.zeros(nq_all, bool)
        valid_q[q0:q0 + len(q)] = ~np.isnan(q).any(1)
        valid_t = np.zeros(nt_all, bool)
        valid_t[t0:t0 + len(t)] = ~np.isnan(t).any(1)
        bmax = float(np.sqrt((ot[:nt_all][valid_t, :dim].astype(np.float64) ** 2).sum(1)).max())
        sub = {x: lists[x] for x in ("kind", "cap")}
        for x in ("cnt", "thr"):
            sub[x] = None if lists[x] is None else lists[x][:, q0:q0 + len(q)]
        for x in ("idx", "val"):
            sub[x] = None if lists[x] is None else lists[x][:, q0:q0 + len(q)]
        check_lists(sub, acc[q0:q0 + len(q)], valid_q[q0:q0 + len(q)], valid_t, na[q0:q0 + len(q)].astype(np.float64),
                    bmax, dim, 5, "batch dim=%d pair %d" % (dim, p), sweep=(t0, t0 + ts[p]), bmax_kernel=bmax_batch)
        q0 += qs[p]
        t0 += ts[p]


# ---- c: adversarial FP16 rounding, black box ---------------------------------------------------------------------------
ULP = 2.0 ** -11          # FP16 spacing in [0.5, 1)


def adversarial_sets(dim, rng, n_zero=16):
    """Source [A; -B], target B: the centre of both sides is exactly 0 (every value is a multiple of 2^-16 below 1,
    so every partial sum the statistics pass forms is exact) and the scale is 1.  A are zero queries; B are one group of
    rows with the same magnitudes w (FP16 grid, [0.5, 1 - 2 ulp]) and random signs:
      5 pushed rows w + (1/2 + i/32) ulp, i = 1..5: FP16 rounds every coordinate AWAY from the query, to w + ulp;
      6 rivals w + ulp on a subset S_j of the coordinates, exact in FP16, with
    |pushed_i|^2 < |rival_j|^2 < |fp16(pushed_i)|^2: the reference's five nearest rows are the pushed ones, the FP16 pass
    ranks all six rivals before them.  B row i sits at target row 32 i, alone in its 32-row chunk (the chunk-entry kernels
    score whole chunks exactly); the other target rows are +-f, f = (1 - ulp) with random signs, alternating, so they
    cancel in the centre and lie beyond every B row.  Returns source, target and the target rows of the pushed rows and
    of the rivals."""
    w = 0.5 + rng.integers(0, 1022, dim) * ULP
    sign = np.where(rng.random(dim) < 0.5, -1.0, 1.0)
    pushed = [sign * (w + (0.5 + i / 32.0) * ULP) for i in range(1, 6)]
    inc = 2 * w * ULP + ULP * ULP                     # what one coordinate at w + ulp adds over w
    e_push = ((w + (0.5 + 5 / 32.0) * ULP) ** 2 - w * w).sum()
    e_fp16 = inc.sum()
    order = rng.permutation(dim)
    pref = np.cumsum(inc[order])
    lo, hi = e_push + 0.02 * (e_fp16 - e_push), e_fp16 - 0.3 * (e_fp16 - e_push)
    cand = np.nonzero((pref > lo) & (pref < hi))[0]
    assert len(cand) >= 6, "dim too small for six rivals"
    picks = cand[np.linspace(0, len(cand) // 3, 6).astype(int)]
    rivals = []
    for m in picks:
        r = w.copy()
        r[order[:m + 1]] += ULP
        rivals.append(sign * r)
    B = np.array(pushed + rivals)
    A = np.zeros((n_zero, dim))
    src = np.concatenate([A, -B]).astype(F32)
    f = np.where(rng.random(dim) < 0.5, -1.0, 1.0) * (1 - ULP)
    n_t = 32 * len(B) + 1
    tgt = np.empty((n_t, dim))
    fill = np.ones(n_t, bool)
    fill[32 * np.arange(len(B))] = False
    tgt[~fill] = B                                     # (-A = A = 0 would sit on the queries)
    tgt[fill] = np.where(np.arange(int(fill.sum()))[:, None] % 2 == 0, f, -f)
    tgt = tgt.astype(F32)
    assert np.array_equal(src.astype(np.float64), np.concatenate([A, -B]))      # exact in FP32
    return src, tgt, 32 * np.arange(5), 32 * np.arange(5, 11)


def twin(src, tgt, dim):
    """CPU twin of the FP16 pass on these sets (centre 0, scale 1): FP16 images and float64 accumulators"""
    a16 = src.astype(np.float16).astype(np.float64)
    b16 = tgt.astype(np.float16).astype(np.float64)
    acc = (b16 ** 2).sum(1)[None, :] - 2 * a16 @ b16.T
    return a16, b16, acc


def margin_use(src, tgt, dim, k):
    """per zero query: (v_nn - T) / (thr_design(T) - T) over the reference's top k, and whether eta = 0 loses one"""
    a16, b16, acc = twin(src, tgt, dim)
    idx, _, _ = orc.knn(src, tgt, k)
    bmax = float(np.sqrt((b16 ** 2).sum(1)).max())
    na = (a16 ** 2).sum(1)
    T = np.sort(acc, axis=1)[:, k - 1]
    v_true = np.take_along_axis(acc, idx.astype(np.int64), axis=1).max(1)
    use = (v_true - T) / (thr_design(T, na, bmax, dim) - T)
    lost_eta0 = v_true >= thr_kernel(T, na, bmax, dim, "eta")
    return use, lost_eta0, v_true < thr_design(T, na, bmax, dim)


C_DIMS = [33, 352, 1960]


@pytest.mark.parametrize("dim", C_DIMS)
def test_adversarial_rounding_twin(dim):
    """CPU: the construction does what it claims, in numpy FP16 and float64 against the oracle's distances"""
    src, tgt, push, riv = adversarial_sets(dim, np.random.default_rng(dim))
    a16, b16, acc = twin(src, tgt, dim)
    assert np.all(b16[push] != tgt[push])                                       # pushed rows round
    assert np.all(np.abs(b16[push]) > np.abs(tgt[push]))                        # ... away from the zero queries
    assert np.array_equal(b16[riv], tgt[riv])                                   # rivals are exact
    assert abs(np.concatenate([src, tgt]).astype(np.float64).sum(0)).max() == 0  # centre 0
    for k in (1, 2, 5):
        idx, _, _ = orc.knn(src, tgt, k)
        assert np.all(idx[:16] == push[:k]), k                                  # reference: the pushed rows
        fp16_rank = np.argsort(acc[0], kind="stable")[:6]
        assert set(fp16_rank.tolist()) == set(riv.tolist()), k                  # FP16: the rivals first
        use, lost, covered = margin_use(src, tgt, dim, k)
        # K-streamed: the step-count slop alone (2 ksteps 2^-21 |b|^2) covers this push, so eta = 0 loses nothing there
        assert np.all(covered) and (k_streamed(dim) or np.any(lost[:16])), (k, use[:16].max())


@gpu
@pytest.mark.parametrize("dim", C_DIMS)
def test_adversarial_rounding_against_the_oracle(dim):
    import torch
    from lidar_global_registration_b200 import device as dev
    src, tgt, push, riv = adversarial_sets(dim, np.random.default_rng(dim))
    exp = {(k, d): orc.knn(*((src, tgt) if d == 0 else (tgt, src)), k) for k in (1, 2, 5) for d in (0, 1)}
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        ops, _, scale = ctx.debug_operands(1, False)
        assert scale == 1.0
        assert ops[:len(tgt), :dim].tobytes() == tgt.astype(np.float16).tobytes()   # rounded as designed (centre 0)
        for k in (1, 2, 5):
            for d in (0, 1):
                ctx.reset_stats()
                _same(ctx.knn(k, d), exp[(k, d)], "knn dim=%d k=%d dir=%d" % (dim, k, d))
                assert ctx.stats()["candidate_launches"] == 1
            for mode, name in ((M.MODE_ONE_SIDED, "one_sided"), (M.MODE_MUTUAL, "mutual"), (M.MODE_RATIO, "ratio")):
                if mode == M.MODE_RATIO and k < 2:
                    continue          # the ratio test needs a second neighbour
                got, avg = ctx.match(k, mode)
                e, eavg = orc.match(src, tgt, k, name, distance_thr=np.float32(M.FLT_MAX))
                assert got.tobytes() == e.tobytes() and avg == eavg, (dim, k, name)
        pairs = [(src, tgt), (tgt, src)]
        for k in (1, 2, 5):
            res = ctx.knn_batch(k, pairs, dim)
            _same(res[0], exp[(k, 0)], "knn_batch")
            _same(res[1], exp[(k, 1)], "knn_batch reverse")
    b = dev.GpuBackend(0)
    tp = [(torch.from_numpy(s).cuda(), torch.from_numpy(t).cuda()) for s, t in pairs]
    for k in (1, 2, 5):
        for p, r in enumerate(b.knn_batch(k, tp, dim)):
            _same([x.cpu().numpy() for x in r], exp[(k, p)], "knn_batch_device k=%d pair %d" % (k, p))
        plan = b.plan_knn_batch(k, tp, dim)
        plan.run()
        for p, r in enumerate(plan.results()):
            _same([x.cpu().numpy() for x in r], exp[(k, p)], "plan k=%d pair %d" % (k, p))
        plan.close()
    b.close()
    for k in (1, 2, 5):
        use, lost, covered = margin_use(src, tgt, dim, k)
        print("dim %d k %d: largest margin use (v_nn - T) / (thr_design(T) - T) = %.3f; eta = 0 loses %d of %d rows"
              % (dim, k, use[:16].max(), lost[:16].sum(), 16))
        assert np.all(covered) and (k_streamed(dim) or np.any(lost[:16]))


# ---- d: A-resident accumulators on adversarial rows ----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dim", [33, 352, 509, 637])
def test_a_resident_accumulators_on_sign_aligned_rows(dim):
    """every column +-1 after centring, signs aligned per row (monotone partial sums): worst error within a quarter of
    the A-resident slop 2^-16 (|a| + |b|)^2 (up to 40 K steps at D = 637)"""
    rng = np.random.default_rng(dim)
    nq, nt = 300, 600
    sgn_q = np.where(rng.random((nq, 1)) < 0.5, -1.0, 1.0)
    sgn_t = np.where(rng.random((nt, 1)) < 0.5, -1.0, 1.0)
    src = (sgn_q * np.ones((nq, dim)) * (1 - 2e-3 * rng.random((nq, dim)))).astype(F32)
    tgt = (sgn_t * np.ones((nt, dim)) * (1 - 2e-3 * rng.random((nt, dim)))).astype(F32)
    assert not k_streamed(dim)
    with M.Context(0) as ctx:
        ctx.upload(0, src, dim)
        ctx.upload(1, tgt, dim)
        oq, _, _ = ctx.debug_operands(0, True)
        ot, _, _ = ctx.debug_operands(1, False)
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
            worst = max(worst, float((err / np.broadcast_to((na + nb) ** 2 + 1e-30, err.shape))[ok].max()))
        ratio = worst / 2.0 ** -16
        print("dim %d (%d K steps): max accumulation error / (|a|+|b|)^2 = %.3e, slop 2^-16 = %.3e, margin %.1fx"
              % (dim, ksteps_of(dim), worst, 2.0 ** -16, 1.0 / max(ratio, 1e-30)))
        assert ratio <= 0.25
        _same(ctx.knn(2, 0), orc.knn(src, tgt, 2))
