"""Batch plans with live counts (b200m_plan_knn_batch_rows / b200m_plan_match_batch_rows through GpuBackend.plan_*(rows=),
b200m_plan_match_multiscale[_local]_batch_rows through plan_match_wide[_local]_batch(kps_rows=, scale_rows=)): a plan is
bound to capacity-sized tensors and int32 tensors of live counts that every run reads.  After every run -- and every replay of one captured torch.cuda.graph -- with counts and rows rewritten in place, the
outputs must be, byte for byte, what the device form (GpuBackend.knn_batch / match_batch) gives on the live prefixes, and
the k-list rows past a live count must hold the empty list.  Rows past the live counts hold NaN, huge values or -inf (and
out-of-range index map entries) and must change nothing.  GPU tests run with -m gpu on a B200; the C-ABI surface is checked without one."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRIES = ["b200m_plan_knn_batch_rows", "b200m_plan_match_batch_rows"]
DTHR = np.float32(0.7)
STALE = [np.float32(np.nan), np.float32(3e38), np.float32(-np.inf), np.float32(1e30)]


def _lib_built():
    return os.path.exists(M._LIB_PATH)


# ---- C-ABI surface (no GPU) -----------------------------------------------------------------------------------------------
def test_rows_entries_exported_declared_and_typed():
    text = open(os.path.join(ROOT, "include", "b200match.h")).read()
    declared = set(re.findall(r"B200M_API\s+[\w\s\*]+?\b(b200m_\w+)\s*\(", text))
    for name in ENTRIES:
        assert name in M.EXPORTS and name in declared, name
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    assert len(L.b200m_plan_knn_batch_rows.argtypes) == 12
    assert len(L.b200m_plan_match_batch_rows.argtypes) == 16


def test_over_capacity_status_text():
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    assert L.b200m_plan_status_error(None, (7 << 16) | 2).decode() == \
        "pair 7, scale 0: the live source row count is above its capacity"
    assert L.b200m_plan_status_error(None, (3 << 16) | 3).decode() == \
        "pair 3, scale 0: the live target row count is above its capacity"
    # the bad-map texts are unchanged
    assert L.b200m_plan_status_error(None, (2 << 48) | (5 << 16) | 1).decode() == \
        "pair 5, scale 2: an index map entry of the target cloud is outside its keypoint range"
    assert L.b200m_plan_status_error(None, 0xFFFFFFFFFFFFFFFF) is None


def test_rows_plan_without_context_fails_loudly():
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    p = M.Context._params(1, M.MODE_MUTUAL)
    pairs = M.Context._device_pairs([(0, 0, 0, 0)])
    h = C.c_void_p(1234)
    assert L.b200m_plan_knn_batch_rows(None, C.byref(p), pairs, 1, 132, 33, None, None, None, None, None, C.byref(h)) != 0
    assert not h.value
    assert L.b200m_plan_last_error(None).decode() == "null context"
    h = C.c_void_p(1234)
    assert L.b200m_plan_match_batch_rows(None, C.byref(p), pairs, 1, 132, 33, None, None, None, 0, None, None, None, None, None,
                                         C.byref(h)) != 0
    assert not h.value


# ---- fixtures and helpers (GPU) -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def backend():
    from lidar_global_registration_b200 import device as D
    b = D.GpuBackend(0)
    yield b
    b.close()


def _caps(B, seed):
    """B (source, target) capacities: the first three fixed (a tile edge, a large pair, a small one), the rest drawn"""
    fixed = [(700, 650), (257, 300), (40, 513)]
    rng = np.random.default_rng(seed)
    return (fixed + [(int(rng.integers(1, 600)), int(rng.integers(1, 600))) for _ in range(B)])[:B]


class Frames:
    """Capacity-sized sets: one device tensor per side holding every pair's slot (3 junk rows between slots), threshold
    tensors split per pair by capacity, and the live counts.  write() rewrites the live rows, fills every row past a live
    count (descriptors and thresholds) with stale values, and sets the counts -- all in place."""

    def __init__(self, dev, desc, caps):
        import torch
        self.torch, self.desc, self.caps = torch, desc, caps
        self.dim, width = synth.DESCRIPTORS[desc]
        self.offs, self.big = [], []
        for side in (0, 1):
            offs, o = [], 0
            for c in caps:
                offs.append(o)
                o += c[side] + 3
            self.offs.append(offs)
            self.big.append(torch.zeros((o, width), dtype=torch.float32, device=dev))
        self.pairs = [(self.big[0][a:a + cs], self.big[1][b:b + ct])
                      for a, b, (cs, ct) in zip(self.offs[0], self.offs[1], caps)]
        self.thr_all = [torch.zeros((sum(c[s] for c in caps),), dtype=torch.float32, device=dev) for s in (0, 1)]
        self.thr = [list(self.thr_all[s].split([c[s] for c in caps])) for s in (0, 1)]
        self.rows = torch.zeros((len(caps), 2), dtype=torch.int32, device=dev)
        self.live = list(caps)

    def write(self, live, seed, scale=1.0):
        torch = self.torch
        stale = STALE[seed % len(STALE)]
        for side in (0, 1):
            self.big[side].fill_(float(stale))
            self.thr_all[side].fill_(float(stale))
        for i, ((ns, nt), (cs, ct)) in enumerate(zip(live, self.caps)):
            ns, nt = min(max(ns, 0), cs), min(max(nt, 0), ct)   # an over-capacity count: the set holds its capacity
            s, t, _ = synth.make_pair(self.desc, max(ns, 1), max(nt, 1), seed=seed * 1000 + i, nan_frac=0.02)
            rng = np.random.default_rng(seed * 1000 + i)
            for side, a, n in ((0, s, ns), (1, t, nt)):
                if n:
                    self.pairs[i][side][:n].copy_(torch.from_numpy(a[:n] * np.float32(scale)))
                    self.thr[side][i][:n].copy_(torch.from_numpy(rng.random(n).astype(np.float32)))
        self.rows.copy_(torch.tensor(live, dtype=torch.int32))
        self.live = [tuple(x) for x in live]

    def live_pairs(self):
        return [(s[:ns], t[:nt]) for (s, t), (ns, nt) in zip(self.pairs, self.live)]

    def live_thr(self):
        return [[self.thr[side][i][:n[side]] for i, n in enumerate(self.live)] for side in (0, 1)]


def _sequence(caps):
    """full capacity; 0 rows on one side; 1 row; counts off and across the 256-row edges; one pair shrinking while another
    grows; every pair empty"""
    def clamp(f):
        return [(max(0, min(cs, a)), max(0, min(ct, b))) for (cs, ct), (a, b) in zip(caps, (f(i, c) for i, c in enumerate(caps)))]
    return [
        ("full", list(caps)),
        ("one side empty", clamp(lambda i, c: (0, c[1]) if i % 2 == 0 else (c[0], 0))),
        ("one row", clamp(lambda i, c: (1, 1))),
        ("tile edges", clamp(lambda i, c: (255 + 2 * (i % 2), 257 - 2 * (i % 2)) if i < 2 else (c[0] - 1, c[1] // 2 + 1))),
        ("shrink and grow", clamp(lambda i, c: (3, 2) if i == 0 else (c[0], c[1]) if i == 1 else (c[0] // 3, c[1] - 1))),
        ("all empty", clamp(lambda i, c: (0, 0))),
    ]


def _check_lists(plan, fr, ref, k, what):
    idx, dist, cnt = plan.idx.cpu().numpy(), plan.dist.cpu().numpy(), plan.cnt.cpu().numpy()
    a = 0
    for p, ((cs, _), (ns, _)) in enumerate(zip(fr.caps, fr.live)):
        if ref is not None:
            for got, r in zip((idx[a:a + ns], dist[a:a + ns], cnt[a:a + ns]), ref[p]):
                assert got.tobytes() == r.cpu().numpy().tobytes(), "%s: pair %d" % (what, p)
        assert (idx[a + ns:a + cs] == -1).all() and (dist[a + ns:a + cs] == 0).all() and (cnt[a + ns:a + cs] == 0).all(), \
            "%s: pair %d rows past the live count" % (what, p)
        a += cs


def _check_records(plan, ref, what):
    got = plan.results()
    for p, ((recs, avg), (rrecs, ravg)) in enumerate(zip(got, ref)):
        assert recs.cpu().numpy().tobytes() == rrecs.cpu().numpy().tobytes(), "%s: pair %d records" % (what, p)
        assert np.float32(avg).tobytes() == np.float32(ravg).tobytes(), "%s: pair %d average" % (what, p)
    assert int(plan.n_out.item()) == sum(r[0].shape[0] for r in ref), what
    assert plan.offsets.cpu().numpy().tolist() == np.cumsum([0] + [r[0].shape[0] for r in ref]).tolist(), what


def _ref_match(b, fr, k, mode, thr):
    kw = {}
    if thr:
        ts, tt = fr.live_thr()
        kw = dict(thr_src=ts, thr_tgt=tt)
    return b.match_batch(k, mode, fr.live_pairs(), fr.dim, distance_thr=DTHR, **kw)


def _plans(b, fr, k):
    """the k-list plan and one match plan per (mode, thresholds) case"""
    cases = [(M.MODE_ONE_SIDED, False), (M.MODE_MUTUAL, False), (M.MODE_MUTUAL, True)]
    if k >= 2:
        cases += [(M.MODE_RATIO, True), (M.MODE_RATIO_MUTUAL, False)]
    pk = b.plan_knn_batch(k, fr.pairs, fr.dim, rows=fr.rows)
    pms = []
    for mode, thr in cases:
        kw = dict(thr_src=fr.thr[0], thr_tgt=fr.thr[1]) if thr else {}
        pms.append((mode, thr, b.plan_match_batch(k, mode, fr.pairs, fr.dim, distance_thr=DTHR, rows=fr.rows, **kw)))
    return pk, pms


def _capture(torch, plans):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for p in plans:
            p.run()
    return g


def _clear(plans):
    for p in plans:
        for name in ("idx", "dist", "cnt", "records", "offsets", "avg", "n_out"):
            t = getattr(p, name, None)
            if t is not None:
                t.fill_(7)


def _check_all(b, fr, k, pk, pms, what):
    ref = b.knn_batch(k, fr.live_pairs(), fr.dim)
    pk.results()   # raises on a set status word
    _check_lists(pk, fr, ref, k, what)
    for mode, thr, pm in pms:
        _check_records(pm, _ref_match(b, fr, k, mode, thr), "%s: mode %d thr %s" % (what, mode, thr))


# ---- the run sequence: runs and replays of one graph ----------------------------------------------------------------------
CASES = [(d, k, B) for d in ("fpfh", "shot") for k in (1, 2, 5) for B in (1, 3, 16)] + [("usc", 1, 3)]


@gpu
@pytest.mark.parametrize("desc,k,B", CASES)
def test_rows_sequence_equals_device_form_on_live_prefixes(backend, desc, k, B):
    import torch
    b = backend
    caps = _caps(B, B * 10 + k)
    if desc == "usc":
        caps = [(300, 260), (257, 1), (40, 200)]
    fr = Frames(b.device, desc, caps)
    seq = _sequence(caps)
    fr.write(seq[0][1], 1)
    pk, pms = _plans(b, fr, k)
    plans = [pk] + [p for _, _, p in pms]
    g = _capture(torch, plans)
    for step, (name, live) in enumerate(seq):
        fr.write(live, step + 2)
        _clear(plans)
        for p in plans:
            p.run()
        _check_all(b, fr, k, pk, pms, "run " + name)
        _clear(plans)
        g.replay()
        _check_all(b, fr, k, pk, pms, "replay " + name)
    for p in plans:
        assert int(p.status.item()) == -1
        p.close()


# ---- over capacity --------------------------------------------------------------------------------------------------------
@gpu
def test_over_capacity_empties_the_pair_and_reports_it(backend):
    import torch
    b = backend
    k = 2
    caps = _caps(3, 5)
    fr = Frames(b.device, "fpfh", caps)
    fr.write(caps, 1)
    pk, pms = _plans(b, fr, k)
    plans = [pk] + [p for _, _, p in pms]
    g = _capture(torch, plans)
    for over, side, text in (((1, 0), 0, "pair 1, scale 0: the live source row count is above its capacity"),
                             ((2, 1), 1, "pair 2, scale 0: the live target row count is above its capacity"),
                             ((0, 0), -1, "pair 0, scale 0: the live source row count is above its capacity")):
        live = [(cs - 5, ct - 3) for cs, ct in caps]
        p_over = over[0]
        if side >= 0:
            live[p_over] = tuple(caps[p_over][s] + 1 if s == side else live[p_over][s] for s in (0, 1))
        else:   # a negative int32 count is far above any capacity
            live[p_over] = (-1, 10)
        fr.write(live, 3 + p_over)
        _clear(plans)
        g.replay()
        torch.cuda.synchronize()
        for p in plans:
            with pytest.raises(M.B200MatchError, match=re.escape(text)):
                p.results()
        # the offending pair answers as empty, every other pair as the device form on its live rows
        fr.live = [(0, 0) if i == p_over else x for i, x in enumerate(live)]
        ref = b.knn_batch(k, fr.live_pairs(), fr.dim)
        _check_lists(pk, fr, ref, k, "over capacity")
        for mode, thr, pm in pms:
            r = _ref_match(b, fr, k, mode, thr)
            offs = pm.offsets.cpu().numpy()
            assert offs.tolist() == np.cumsum([0] + [x[0].shape[0] for x in r]).tolist()
            assert offs[p_over + 1] == offs[p_over]
            recs = pm.records.cpu().numpy()
            for i, (rr, ravg) in enumerate(r):
                assert recs[offs[i]:offs[i + 1]].tobytes() == rr.cpu().numpy().tobytes()
            assert pm.avg.cpu().numpy().tobytes() == np.array([x[1] for x in r], np.float32).tobytes()
            assert np.float32(pm.avg[p_over].item()) == np.float32(M.FLT_MAX)
        # the next valid replay reports clean
        fr.write([(cs // 2, ct // 2) for cs, ct in caps], 9)
        g.replay()
        _check_all(b, fr, k, pk, pms, "after over capacity")
        for p in plans:
            assert int(p.status.item()) == -1
    for p in plans:
        p.close()


@gpu
def test_creation_with_an_over_capacity_count_fails_with_the_text(backend):
    b = backend
    caps = _caps(3, 6)
    fr = Frames(b.device, "fpfh", caps)
    fr.write(caps, 1)
    fr.rows[2, 1] = caps[2][1] + 1
    with pytest.raises(M.B200MatchError, match=re.escape("b200m_plan_knn_batch_rows: pair 2, scale 0: the live target row "
                                                         "count is above its capacity")):
        b.plan_knn_batch(1, fr.pairs, fr.dim, rows=fr.rows)
    with pytest.raises(M.B200MatchError, match=re.escape("b200m_plan_match_batch_rows: pair 2, scale 0: the live target row "
                                                         "count is above its capacity")):
        b.plan_match_batch(1, M.MODE_MUTUAL, fr.pairs, fr.dim, rows=fr.rows)
    with pytest.raises(M.B200MatchError, match="rows: must be"):
        b.plan_knn_batch(1, fr.pairs, fr.dim, rows=fr.rows.long())


# ---- routing on the device ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("desc", ["fpfh", "shot"])
def test_out_of_window_run_then_in_window_run(backend, desc):
    """one run whose live data lies outside the certificate's window (x 1e20: the exact path), then one inside it (the
    tensor cores): both byte-equal to the device form, which takes the same routes"""
    import torch
    b = backend
    caps = _caps(3, 7)
    fr = Frames(b.device, desc, caps)
    fr.write(caps, 1)
    pk, pms = _plans(b, fr, 2)
    g = _capture(torch, [pk] + [p for _, _, p in pms])
    for step, (scale, inside) in enumerate(((1e20, False), (1.0, True))):
        live = [(cs - 17 * step, ct - 9) for cs, ct in caps]
        fr.write(live, 20 + step, scale=scale)
        g.replay()
        _check_all(b, fr, 2, pk, pms, "scale %g" % scale)
        b.ctx.set_profiling(True)
        b.ctx.reset_stats()
        b.knn_batch(2, fr.live_pairs(), fr.dim)
        launches = b.ctx.stats()["candidate_launches"]
        b.ctx.set_profiling(False)
        assert (launches > 0) == inside
    pk.close()
    for _, _, p in pms:
        p.close()


# ---- matcher-class plans with live counts ---------------------------------------------------------------------------------
WIDE_ENTRIES = ["b200m_plan_match_multiscale_batch_rows", "b200m_plan_match_multiscale_local_batch_rows"]
WMODES = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "cluster": M.MODE_CLUSTER}
RADIUS = 0.3
MASK = 0xFFFFFFFFFFFFFFFF
BAD_MAP = [np.int32(1 << 30), np.int32(-7)]   # stale map entries past the live rows: out of any keypoint range


def test_wide_rows_entries_exported_declared_and_typed():
    text = open(os.path.join(ROOT, "include", "b200match.h")).read()
    declared = set(re.findall(r"B200M_API\s+[\w\s\*]+?\b(b200m_\w+)\s*\(", text))
    for name in WIDE_ENTRIES:
        assert name in M.EXPORTS and name in declared, name
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    assert len(L.b200m_plan_match_multiscale_batch_rows.argtypes) == 19
    assert len(L.b200m_plan_match_multiscale_local_batch_rows.argtypes) == 21
    assert L.b200m_plan_status_error(None, (0xFFFF << 48) | (4 << 16) | 2).decode() == \
        "pair 4: the live source keypoint count is above its capacity"
    assert L.b200m_plan_status_error(None, (1 << 48) | (2 << 16) | 3).decode() == \
        "pair 2, scale 1: the live target row count is above its capacity"


def _wide_caps(B, seed):
    """per pair: (source keypoints, target keypoints, [(source rows, target rows) per scale]) capacities"""
    fixed = [(600, 650, [(560, 620), (500, 600), (300, 280)]), (300, 320, [(300, 300), (280, 290)]), (200, 150, [(180, 150)])]
    rng = np.random.default_rng(seed)
    for _ in range(B):
        ns, nt = int(rng.integers(40, 320)), int(rng.integers(40, 320))
        fixed.append((ns, nt, [(int(rng.integers(1, ns + 1)), int(rng.integers(1, nt + 1))) for _ in range(2)]))
    return fixed[:B]


class WideFrames:
    """Capacity-sized matcher-class inputs: per pair and scale a descriptor tensor and an index map, per pair keypoints and
    moved keypoints, threshold tensors split per pair by keypoint capacity, and the two live-count tensors.  write() fills
    everything past a live count with stale values (NaN / huge descriptors and coordinates, out-of-range map entries) and
    the live prefixes with fresh data, all in place."""

    def __init__(self, dev, desc, caps):
        import torch
        self.torch, self.desc, self.caps = torch, desc, caps
        self.dim, width = synth.DESCRIPTORS[desc]
        rng = np.random.default_rng(len(caps))
        t = lambda n, w, dt=torch.float32: torch.zeros((n, w), dtype=dt, device=dev)
        self.pairs = []
        for ck_s, ck_t, rows in caps:
            sc = {"src_scales": [], "tgt_scales": []}
            for rs, rt in rows:
                sc["src_scales"].append((t(rs, width), torch.zeros((rs,), dtype=torch.int32, device=dev)))
                sc["tgt_scales"].append((t(rt, width), torch.zeros((rt,), dtype=torch.int32, device=dev)))
            self.pairs.append(dict(sc, src_kps_xyz=t(ck_s, 4), tgt_kps_xyz=t(ck_t, 4), src_kps_moved=t(ck_s, 4),
                                   tgt_kps_moved=t(ck_t, 4), iss_radius_src=float(0.03 + 0.05 * rng.random()),
                                   iss_radius_tgt=float(0.03 + 0.05 * rng.random())))
        self.thr_all = [torch.zeros((sum(c[s] for c in caps),), dtype=torch.float32, device=dev) for s in (0, 1)]
        self.thr = [list(self.thr_all[s].split([c[s] for c in caps])) for s in (0, 1)]
        self.kps = torch.zeros((len(caps), 2), dtype=torch.int32, device=dev)
        self.rows = torch.zeros((sum(len(c[2]) for c in caps), 2), dtype=torch.int32, device=dev)
        self.live = None

    def write(self, live, seed, scale=1.0):
        """live: per pair (source keypoints, target keypoints, [(source rows, target rows) per scale])"""
        import test_gpu_wide_plan as TW
        torch = self.torch
        rng = np.random.default_rng(seed)
        put = lambda dst, a: dst.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        stale, bad = STALE[seed % len(STALE)], BAD_MAP[seed % len(BAD_MAP)]
        for side in (0, 1):
            self.thr_all[side].fill_(float(stale))
        for i, ((ck_s, ck_t, crows), (ns, nt, rows), pr) in enumerate(zip(self.caps, live, self.pairs)):
            ns, nt = min(max(ns, 0), ck_s), min(max(nt, 0), ck_t)
            for key in ("src_kps_xyz", "tgt_kps_xyz", "src_kps_moved", "tgt_kps_moved"):
                pr[key].fill_(float(stale))
            for s, ((rs, rt), (cs, ct)) in enumerate(zip(rows, crows)):
                rs, rt = min(max(rs, 0), cs), min(max(rt, 0), ct)
                src, tgt, _ = synth.make_pair(self.desc, max(rs, 1), max(rt, 1), seed=1000 * seed + 10 * i + s, nan_frac=0.02)
                for side, n, nk, a in (("src_scales", rs, ns, src), ("tgt_scales", rt, nt, tgt)):
                    f, m = pr[side][s]
                    f.fill_(float(stale))
                    m.fill_(int(bad))
                    if n:
                        put(f[:n], a[:n] * np.float32(scale))
                        # injective, as the scatter needs (two rows of one scale on one keypoint race); more rows than
                        # keypoints only in a pair whose counts are over capacity, which is never read
                        put(m[:n], (rng.permutation(max(nk, n, 1))[:n] % max(nk, 1)).astype(np.int32))
            sx, tx = TW._xyz(rng, ns), TW._xyz(rng, nt)
            g = np.eye(4, dtype=np.float32)
            g[:3, 3] = 0.05 * rng.standard_normal(3)
            if ns:
                put(pr["src_kps_xyz"][:ns], sx)
                put(pr["src_kps_moved"][:ns], M.transform_keypoints(sx, g))
                put(self.thr[0][i][:ns], rng.random(ns).astype(np.float32))
            if nt:
                put(pr["tgt_kps_xyz"][:nt], tx)
                put(pr["tgt_kps_moved"][:nt], M.transform_keypoints(tx, M.invert_guess(g)))
                put(self.thr[1][i][:nt], rng.random(nt).astype(np.float32))
        self.kps.copy_(torch.tensor([(x[0], x[1]) for x in live], dtype=torch.int32))
        self.rows.copy_(torch.tensor([r for x in live for r in x[2]], dtype=torch.int32).reshape(-1, 2))
        self.live = live

    def live_pairs(self):
        out = []
        for (ns, nt, rows), pr in zip(self.live, self.pairs):
            d = dict(pr)
            for side, j in (("src_scales", 0), ("tgt_scales", 1)):
                d[side] = [(f[:r[j]], m[:r[j]]) for (f, m), r in zip(pr[side], rows)]
            for key, n in (("src_kps_xyz", ns), ("src_kps_moved", ns), ("tgt_kps_xyz", nt), ("tgt_kps_moved", nt)):
                d[key] = pr[key][:n]
            out.append(d)
        return out

    def live_thr(self):
        return [[self.thr[side][i][:x[side]] for i, x in enumerate(self.live)] for side in (0, 1)]


def _wide_sequence(caps):
    """full capacity; 0 keypoints (a pair without source keypoints, one without target keypoints); 1 keypoint and 1 row;
    rows off and across the 256-row edges; one pair shrinking while another grows; every pair empty"""
    def clamp(f):
        out = []
        for i, c in enumerate(caps):
            ns, nt, rows = f(i, c)
            ns, nt = max(0, min(c[0], ns)), max(0, min(c[1], nt))
            rows = [(max(0, min(cs, rs, ns)), max(0, min(ct, rt, nt))) for (cs, ct), (rs, rt) in zip(c[2], rows)]
            out.append((ns, nt, rows))
        return out
    return [
        ("full", clamp(lambda i, c: (c[0], c[1], c[2]))),
        ("0 keypoints", clamp(lambda i, c: (0 if i % 2 == 0 else c[0], c[1] if i % 2 == 0 else 0, c[2]))),
        ("one row", clamp(lambda i, c: (1, 1, [(1, 1)] * len(c[2])))),
        ("tile edges", clamp(lambda i, c: (c[0] - 1, c[1] - 2, [(255 + 2 * (s % 2), 257 - 2 * (s % 2)) if i == 0 else
                                                               (r[0] - 1, r[1] // 2 + 1) for s, r in enumerate(c[2])]))),
        ("shrink and grow", clamp(lambda i, c: ((5, 4, [(3, 2)] * len(c[2])) if i == 0 else (c[0], c[1], c[2]) if i == 1 else
                                                (c[0] // 3, c[1] - 1, [(r[0] // 3, r[1] - 1) for r in c[2]])))),
        ("all empty", clamp(lambda i, c: (0, 0, [(0, 0)] * len(c[2])))),
    ]


def _wide_arms(guessed=(False, True)):
    return [(m, gs, th) for m in WMODES for gs in guessed for th in (False, True)]


def _wide_call(b, wf, k, m, gs, th, plan=False):
    kw = dict(dim=wf.dim, distance_thr=DTHR)
    if plan:
        kw.update(kps_rows=wf.kps, scale_rows=wf.rows)
        if th:
            kw.update(thr_src=wf.thr[0], thr_tgt=wf.thr[1])
        pairs = wf.pairs
    else:
        if th:
            ts, tt = wf.live_thr()
            kw.update(thr_src=ts, thr_tgt=tt)
        pairs = wf.live_pairs()
    if gs:
        f = b.plan_match_wide_local_batch if plan else b.match_wide_local_batch
        return f(k, WMODES[m], pairs, RADIUS, **kw)
    f = b.plan_match_wide_batch if plan else b.match_wide_batch
    return f(k, WMODES[m], pairs, **kw)


def _wide_same(plan, ref, what):
    got = plan.results()
    assert int(plan.status.item()) & MASK == MASK, what
    for p, ((recs, avg), (rrecs, ravg)) in enumerate(zip(got, ref)):
        assert recs.cpu().numpy().tobytes() == rrecs.cpu().numpy().tobytes(), "%s: pair %d records" % (what, p)
        assert np.float32(avg).tobytes() == np.float32(ravg).tobytes(), "%s: pair %d average" % (what, p)
    assert int(plan.n_out.item()) == sum(r[0].shape[0] for r in ref), what
    assert plan.offsets.cpu().numpy().tolist() == np.cumsum([0] + [r[0].shape[0] for r in ref]).tolist(), what


def _wide_check_all(b, wf, k, arms, plans, what):
    for (m, gs, th), p in zip(arms, plans):
        _wide_same(p, _wide_call(b, wf, k, m, gs, th), "%s: %s guessed=%s thr=%s" % (what, m, gs, th))


WIDE_CASES = [("fpfh", 1, 1), ("fpfh", 2, 3), ("shot", 2, 3), ("fpfh", 2, 16), ("usc", 1, 3)]


@gpu
@pytest.mark.parametrize("desc,k,B", WIDE_CASES)
def test_wide_rows_sequence_equals_device_form_on_live_prefixes(backend, desc, k, B):
    """OneSided / LeftToRight / Cluster, guessed and not, with and without thresholds: every run and every replay of one
    captured graph equals the device form on the live prefixes"""
    import torch
    b = backend
    caps = _wide_caps(B, 40 + B)
    if desc == "usc":
        caps = [(120, 130, [(120, 130), (100, 110)]), (90, 100, [(90, 100)]), (257, 255, [(257, 255), (256, 200)])]
    wf = WideFrames(b.device, desc, caps)
    seq = _wide_sequence(caps)
    wf.write(seq[0][1], 1)
    arms = _wide_arms()
    plans = [_wide_call(b, wf, k, m, gs, th, plan=True) for m, gs, th in arms]
    g = _capture(torch, plans)
    for step, (name, live) in enumerate(seq):
        wf.write(live, step + 2)
        _clear(plans)
        for p in plans:
            p.run()
        _wide_check_all(b, wf, k, arms, plans, "run " + name)
        _clear(plans)
        g.replay()
        _wide_check_all(b, wf, k, arms, plans, "replay " + name)
    for p in plans:
        p.close()


@gpu
def test_wide_over_capacity_empties_the_pair_and_reports_it(backend):
    import torch
    b = backend
    k = 2
    caps = _wide_caps(3, 9)
    wf = WideFrames(b.device, "fpfh", caps)
    full = [(c[0], c[1], list(c[2])) for c in caps]
    wf.write(full, 1)
    arms = _wide_arms()
    plans = [_wide_call(b, wf, k, m, gs, th, plan=True) for m, gs, th in arms]
    g = _capture(torch, plans)
    half = [(c[0] // 2, c[1] // 2, [(r[0] // 2, r[1] // 2) for r in c[2]]) for c in caps]
    cases = [(1, lambda x, c: (c[0] + 1, x[1], x[2]), "pair 1: the live source keypoint count is above its capacity"),
             (0, lambda x, c: (x[0], x[1], [x[2][0], (x[2][1][0], c[2][1][1] + 1)] + x[2][2:]),
              "pair 0, scale 1: the live target row count is above its capacity"),
             (2, lambda x, c: (x[0], -1, x[2]), "pair 2: the live target keypoint count is above its capacity")]
    for p_over, bump, text in cases:
        live = list(half)
        live[p_over] = bump(half[p_over], caps[p_over])
        wf.write(live, 5 + p_over)
        _clear(plans)
        g.replay()
        torch.cuda.synchronize()
        for p in plans:
            with pytest.raises(M.B200MatchError, match=re.escape(text)):
                p.results()
        # the offending pair answers as empty, every other pair as the device form on its live rows
        wf.live = [(0, 0, [(0, 0)] * len(x[2])) if i == p_over else x for i, x in enumerate(live)]
        for (m, gs, th), p in zip(arms, plans):
            ref = _wide_call(b, wf, k, m, gs, th)
            offs = p.offsets.cpu().numpy()
            assert offs.tolist() == np.cumsum([0] + [r[0].shape[0] for r in ref]).tolist()
            assert offs[p_over + 1] == offs[p_over]
            recs = p.records.cpu().numpy()
            for i, (rr, _ravg) in enumerate(ref):
                assert recs[offs[i]:offs[i + 1]].tobytes() == rr.cpu().numpy().tobytes()
            assert p.avg.cpu().numpy().tobytes() == np.array([r[1] for r in ref], np.float32).tobytes()
        wf.write(half, 11)
        g.replay()
        _wide_check_all(b, wf, k, arms, plans, "after over capacity")
    bad = list(full)
    bad[1] = (caps[1][0] + 5, caps[1][1], caps[1][2])
    wf.write(bad, 12)
    with pytest.raises(M.B200MatchError, match=re.escape("b200m_plan_match_multiscale_batch_rows: pair 1: the live source "
                                                         "keypoint count is above its capacity")):
        _wide_call(b, wf, k, "mutual", False, False, plan=True)
    for p in plans:
        p.close()


@gpu
@pytest.mark.parametrize("desc", ["fpfh", "shot"])
def test_wide_out_of_window_run_then_in_window_run(backend, desc):
    import torch
    b = backend
    caps = _wide_caps(3, 13)
    wf = WideFrames(b.device, desc, caps)
    wf.write([(c[0], c[1], list(c[2])) for c in caps], 1)
    arms = _wide_arms(guessed=(False,))
    plans = [_wide_call(b, wf, 2, m, gs, th, plan=True) for m, gs, th in arms]
    g = _capture(torch, plans)
    for step, scale in enumerate((1e20, 1.0)):
        live = [(c[0] - 3 * step, c[1] - 5, [(min(r[0] - 7, c[0] - 3 * step), min(r[1] - 2 * step, c[1] - 5)) for r in c[2]])
                for c in caps]
        wf.write(live, 30 + step, scale=scale)
        g.replay()
        _wide_check_all(b, wf, 2, arms, plans, "scale %g" % scale)
    for p in plans:
        p.close()
