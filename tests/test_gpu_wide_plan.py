"""Matcher-class batch plans (b200m_plan_match_multiscale_batch / b200m_plan_match_multiscale_local_batch through
GpuBackend.plan_match_wide_batch / plan_match_wide_local_batch): OneSided / LeftToRight / Cluster batches, guessed or not,
bound once and captured in torch.cuda.graph (global capture mode: a sync, an allocation or a pageable copy inside run would
fail the capture).  After every bound input -- descriptors, maps, coordinates, moved coordinates, thresholds -- is rewritten
in place, a replay must give, byte for byte, what the device form (GpuBackend.match_wide_batch / match_wide_local_batch)
gives on the new data: outside the certificate's window too, with a bad map entry (the status word), with a capacity below
the records found, and after the caller's own context has grown its workspaces.  GPU tests run with -m gpu on a B200; the
C-ABI surface is checked without one."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDE_PLAN_ENTRIES = ["b200m_plan_match_multiscale_batch", "b200m_plan_match_multiscale_local_batch", "b200m_plan_status_error"]
WMODES = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "cluster": M.MODE_CLUSTER}
DTHR = np.float32(0.7)
RADIUS = 0.3
MASK = 0xFFFFFFFFFFFFFFFF


def _lib_built():
    return os.path.exists(M._LIB_PATH)


# ---- C-ABI surface (no GPU) -----------------------------------------------------------------------------------------------
def test_wide_plan_entries_exported_and_declared():
    text = open(os.path.join(ROOT, "include", "b200match.h")).read()
    declared = set(re.findall(r"B200M_API\s+[\w\s\*]+?\b(b200m_\w+)\s*\(", text))
    for name in WIDE_PLAN_ENTRIES:
        assert name in M.EXPORTS, name
        assert name in declared, name


def test_wide_plan_entries_have_argtypes():
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    assert len(L.b200m_plan_match_multiscale_batch.argtypes) == 17
    assert len(L.b200m_plan_match_multiscale_local_batch.argtypes) == 19
    assert len(L.b200m_plan_status_error.argtypes) == 2
    assert L.b200m_plan_status_error.restype is C.c_char_p


def test_status_text_needs_no_device():
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    assert L.b200m_plan_status_error(None, MASK) is None
    key = (3 << 48) | (17 << 16) | 1
    assert L.b200m_plan_status_error(None, key).decode() == \
        "pair 17, scale 3: an index map entry of the target cloud is outside its keypoint range"
    assert L.b200m_plan_status_error(None, 2 << 16).decode() == \
        "pair 2, scale 0: an index map entry of the source cloud is outside its keypoint range"


def test_wide_plan_without_context_fails_loudly():
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    p = M.Context._params(1, M.MODE_MUTUAL)
    arr, locs, _keep = M.Context._wide_device_pairs([dict(scales=[], n_src_kps=0, n_tgt_kps=0, iss_radius_src=0.05,
                                                          iss_radius_tgt=0.05)], True)
    h = C.c_void_p(1234)
    assert L.b200m_plan_match_multiscale_batch(None, C.byref(p), arr, 1, 132, 33, 16, 40, None, None, None, 0, None, None, None,
                                               None, C.byref(h)) != 0
    assert not h.value
    assert L.b200m_plan_last_error(None).decode() == "null context"
    h = C.c_void_p(1234)
    assert L.b200m_plan_match_multiscale_local_batch(None, C.byref(p), arr, locs, 1, 132, 33, 16, 40, 0.3, None, None, None, 0,
                                                     None, None, None, None, C.byref(h)) != 0
    assert not h.value
    assert L.b200m_plan_last_error(None).decode() == "null context"


# ---- fixtures and helpers (GPU) -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def backend():
    from lidar_global_registration_b200 import device as D
    b = D.GpuBackend(0)
    yield b
    b.close()


def _xyz(rng, n):
    x = np.zeros((n, 4), np.float32)
    x[:, :3] = rng.random((n, 3)) * 4
    if n:
        x[: n // 4, :3] = x[0, :3] + 0.02 * rng.standard_normal((n // 4, 3)).astype(np.float32)
    return x


def _spec(n_sk, n_tk, rows, null=()):
    """one pair: keypoints per side, rows per scale, and the scales whose maps are NULL (then rows == keypoints)"""
    return dict(n_sk=n_sk, n_tk=n_tk, rows=rows, null=set(null))


# the batch of every capture test: every scale set size at the 255 / 256 / 257-row edges, NULL maps, a pair without source
# keypoints, one with fewer scales, one without target keypoints, and a last pair aliasing the first one's tensors
SPECS = {
    "long": [_spec(600, 700, [(600, 700), (550, 660), (500, 620)], null=[0]),
             _spec(300, 300, [(255, 257), (256, 256), (257, 255)]),
             _spec(0, 300, [(0, 300)] * 3),
             _spec(400, 450, [(400, 450), (380, 420)], null=[0]),
             _spec(350, 0, [(350, 0)] * 3, null=[0, 1, 2])],
    "usc": [_spec(120, 130, [(120, 130), (100, 110)], null=[0]),
            _spec(0, 90, [(0, 90)] * 2),
            _spec(90, 100, [(90, 100)]),
            _spec(257, 255, [(257, 255), (256, 200)], null=[0])],
}


class WideBound:
    """Device tensors for a batch of pair specs (every descriptor set, map, keypoint and moved keypoint table its own
    tensor; the last pair aliases the first), threshold tensors split per pair, and the dicts GpuBackend takes.  write()
    rewrites every one of them in place."""

    def __init__(self, dev, desc, specs, seed):
        import torch
        self.torch, self.desc, self.specs = torch, desc, specs
        self.dim = synth.DESCRIPTORS[desc][0]
        width = synth.make_pair(desc, 1, 1, seed=0)[0].shape[1]
        rng = np.random.default_rng(seed)
        self.pairs = []
        for sp in specs:
            t = lambda n, w, dt=torch.float32: torch.zeros((n, w), dtype=dt, device=dev)
            sc = {"src_scales": [], "tgt_scales": []}
            for s, (ns, nt) in enumerate(sp["rows"]):
                for side, n, nk in (("src_scales", ns, sp["n_sk"]), ("tgt_scales", nt, sp["n_tk"])):
                    m = None if s in sp["null"] or n == 0 else torch.zeros((n,), dtype=torch.int32, device=dev)
                    sc[side].append((t(n, width), m))
            self.pairs.append(dict(sc, src_kps_xyz=t(sp["n_sk"], 4), tgt_kps_xyz=t(sp["n_tk"], 4), src_kps_moved=t(sp["n_sk"], 4),
                                   tgt_kps_moved=t(sp["n_tk"], 4), iss_radius_src=float(0.03 + 0.05 * rng.random()),
                                   iss_radius_tgt=float(0.03 + 0.05 * rng.random())))
        self.pairs.append(self.pairs[0])
        counts = [(pr["src_kps_xyz"].shape[0], pr["tgt_kps_xyz"].shape[0]) for pr in self.pairs]
        self.thr_all = [torch.zeros((sum(c[s] for c in counts),), dtype=torch.float32, device=dev) for s in (0, 1)]
        self.thr = [list(self.thr_all[s].split([c[s] for c in counts])) for s in (0, 1)]
        self.write(seed)

    def write(self, seed):
        torch = self.torch
        rng = np.random.default_rng(seed)
        put = lambda dst, a: dst.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        for i, (sp, pr) in enumerate(zip(self.specs, self.pairs)):
            for s, (ns, nt) in enumerate(sp["rows"]):
                src, tgt, _ = synth.make_pair(self.desc, max(ns, 1), max(nt, 1), seed=1000 * seed + 10 * i + s, nan_frac=0.02)
                for side, n, nk, a in (("src_scales", ns, sp["n_sk"], src), ("tgt_scales", nt, sp["n_tk"], tgt)):
                    f, m = pr[side][s]
                    put(f, a[:n])
                    if m is not None:
                        put(m, np.sort(rng.choice(nk, n, replace=False)).astype(np.int32))
            sx, tx = _xyz(rng, sp["n_sk"]), _xyz(rng, sp["n_tk"])
            g = np.eye(4, dtype=np.float32)
            g[:3, 3] = 0.05 * rng.standard_normal(3)
            put(pr["src_kps_xyz"], sx)
            put(pr["tgt_kps_xyz"], tx)
            put(pr["src_kps_moved"], M.transform_keypoints(sx, g))
            put(pr["tgt_kps_moved"], M.transform_keypoints(tx, M.invert_guess(g)))
        for side in (0, 1):
            put(self.thr_all[side], rng.random(self.thr_all[side].shape[0]).astype(np.float32))


def _capture(torch, plans):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for p in plans:
            p.run()
    return g


def _same_records(plan, ref):
    got = plan.results()
    assert int(plan.status.item()) & MASK == MASK
    assert len(got) == len(ref)
    for p, ((recs, avg), (rrecs, ravg)) in enumerate(zip(got, ref)):
        assert recs.cpu().numpy().tobytes() == rrecs.cpu().numpy().tobytes(), "pair %d records" % p
        assert np.float32(avg).tobytes() == np.float32(ravg).tobytes(), "pair %d average" % p
    assert int(plan.n_out.item()) == sum(r[0].shape[0] for r in ref)
    assert plan.offsets.cpu().numpy().tolist() == np.cumsum([0] + [r[0].shape[0] for r in ref]).tolist()


class Arms:
    """every (mode, guessed, thresholds) plan of a bound batch, and the device-form call each one must equal"""

    def __init__(self, b, bd, k, guessed=(False, True), thresholds=(False, True), modes=tuple(WMODES)):
        self.b, self.bd, self.k = b, bd, k
        self.arms = [(m, gs, th) for m in modes for gs in guessed for th in thresholds]
        self.plans = [self._call(m, gs, th, plan=True) for m, gs, th in self.arms]

    def _call(self, m, gs, th, plan=False, **extra):
        b, bd = self.b, self.bd
        kw = dict(dim=bd.dim, distance_thr=DTHR, **extra)
        if th:
            kw.update(thr_src=bd.thr[0], thr_tgt=bd.thr[1])
        if gs:
            f = b.plan_match_wide_local_batch if plan else b.match_wide_local_batch
            return f(self.k, WMODES[m], bd.pairs, RADIUS, **kw)
        f = b.plan_match_wide_batch if plan else b.match_wide_batch
        return f(self.k, WMODES[m], bd.pairs, **kw)

    def check(self):
        for (m, gs, th), p in zip(self.arms, self.plans):
            try:
                _same_records(p, self._call(m, gs, th))
            except AssertionError as e:
                raise AssertionError("%s guessed=%s thresholds=%s: %s" % (m, gs, th, e))

    def close(self):
        for p in self.plans:
            p.close()


# ---- capture, rewrite and replay ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("desc,k", [("fpfh", 1), ("fpfh", 2), ("shot", 2), ("usc", 1)])
def test_capture_and_replay_equals_device_form(backend, desc, k):
    import torch
    bd = WideBound(backend.device, desc, SPECS["usc" if desc == "usc" else "long"], 1)
    arms = Arms(backend, bd, k)
    arms.check()                       # the creation run
    g = _capture(torch, arms.plans)
    for seed in (2, 3):
        bd.write(seed)
        g.replay()
        arms.check()
    arms.close()


# ---- routing on the device ------------------------------------------------------------------------------------------------
@gpu
def test_replay_outside_the_window_equals_device_form(backend):
    """one scale's descriptors at 1e19 (beyond the certificate's upper edge at dim 33): the device form sends that scale to
    the exact path on the host's decision, a replay on the device's; then ordinary data again"""
    import torch
    bd = WideBound(backend.device, "fpfh", SPECS["long"], 4)
    arms = Arms(backend, bd, 2, guessed=(False,), thresholds=(False,))
    g = _capture(torch, arms.plans)
    bd.write(5)
    for pr in bd.pairs[:-1]:
        for side in ("src_scales", "tgt_scales"):
            if len(pr[side]) > 1:
                pr[side][1][0].mul_(1e19)
    g.replay()
    arms.check()
    bd.write(6)
    g.replay()
    arms.check()
    arms.close()


# ---- the status word ------------------------------------------------------------------------------------------------------
@gpu
def test_status_names_the_bad_map_entry_and_clears(backend):
    import torch
    bd = WideBound(backend.device, "fpfh", SPECS["long"], 7)
    arms = Arms(backend, bd, 2, thresholds=(False,), modes=("mutual", "cluster"))
    g = _capture(torch, arms.plans)
    smap = bd.pairs[1]["src_scales"][1][1]
    saved = smap.clone()
    smap[7] = 10 ** 6
    g.replay()
    key = (1 << 48) | (1 << 16) | 0
    for (m, gs, _), p in zip(arms.arms, arms.plans):
        torch.cuda.synchronize()
        assert int(p.status.item()) & MASK == key, (m, gs)
        with pytest.raises(M.B200MatchError) as ed:
            arms._call(m, gs, False)
        text = str(ed.value)
        assert text.endswith("pair 1, scale 1: an index map entry of the source cloud is outside its keypoint range"), text
        with pytest.raises(M.B200MatchError) as ep:
            p.results()
        assert text.endswith(": " + str(ep.value)), (text, str(ep.value))
    smap.copy_(saved)
    g.replay()
    arms.check()
    arms.close()


@gpu
def test_creation_with_a_bad_map_fails_with_the_device_text(backend):
    bd = WideBound(backend.device, "fpfh", SPECS["long"], 8)
    bd.pairs[3]["tgt_scales"][1][1][0] = -1
    with pytest.raises(M.B200MatchError) as ed:
        backend.match_wide_batch(2, M.MODE_MUTUAL, bd.pairs, bd.dim)
    with pytest.raises(M.B200MatchError) as ep:
        backend.plan_match_wide_batch(2, M.MODE_MUTUAL, bd.pairs, bd.dim)
    assert str(ed.value) == str(ep.value).replace("b200m_plan_match_multiscale_batch", "b200m_match_multiscale_batch_device")
    assert "pair 3, scale 1: an index map entry of the target cloud" in str(ep.value)


# ---- capacity and ownership -----------------------------------------------------------------------------------------------
@gpu
def test_capacity_is_reported_not_enforced(backend):
    import torch
    bd = WideBound(backend.device, "fpfh", SPECS["long"], 9)
    ref = backend.match_wide_batch(2, M.MODE_CLUSTER, bd.pairs, bd.dim)
    n = sum(r[0].shape[0] for r in ref)
    assert n > 10
    cap = n // 3
    p = backend.plan_match_wide_batch(2, M.MODE_CLUSTER, bd.pairs, bd.dim, cap=cap)
    p.records.zero_()
    p.run()
    torch.cuda.synchronize()
    assert int(p.n_out.item()) == n and int(p.status.item()) & MASK == MASK
    full = torch.cat([r[0] for r in ref])
    assert p.records.cpu().numpy().tobytes() == full[:cap].cpu().numpy().tobytes()
    assert p.offsets.cpu().numpy().tolist() == np.cumsum([0] + [r[0].shape[0] for r in ref]).tolist()
    assert p.avg.cpu().numpy().tobytes() == np.array([r[1] for r in ref], np.float32).tobytes()
    with pytest.raises(M.B200MatchError, match="capacity"):
        p.results()
    p.close()


@gpu
def test_caller_context_growth_does_not_move_the_plan(backend):
    import torch
    bd = WideBound(backend.device, "shot", SPECS["long"], 11)
    arms = Arms(backend, bd, 2, thresholds=(True,))
    g = _capture(torch, arms.plans)
    big = WideBound(backend.device, "shot", [_spec(3000, 3500, [(3000, 3500), (2900, 3300)]),
                                             _spec(2600, 2900, [(2600, 2900), (2500, 2800)])], 12)
    backend.match_wide_batch(2, M.MODE_CLUSTER, big.pairs, big.dim)
    backend.match_wide_local_batch(5, M.MODE_MUTUAL, big.pairs, RADIUS, big.dim)
    bd.write(13)
    g.replay()
    arms.check()
    arms.close()


@gpu
def test_refusals_and_batches_without_source_keypoints(backend):
    import torch
    b = backend
    src, tgt, dim = synth.make_pair("fpfh", 300, 300, seed=14, nan_frac=0.0)
    ds, dt = torch.from_numpy(src).to(b.device), torch.from_numpy(tgt).to(b.device)
    xyz = torch.zeros((300, 4), dtype=torch.float32, device=b.device)
    hmap = np.arange(300, dtype=np.int32)
    wide = dict(scales=[(ds.data_ptr(), 300, 0, dt.data_ptr(), 300, 0)], n_src_kps=300, n_tgt_kps=300,
                src_kps_xyz=xyz.data_ptr(), tgt_kps_xyz=xyz.data_ptr(), iss_radius_src=0.05, iss_radius_tgt=0.05)
    bad = dict(wide, scales=[wide["scales"][0], (ds.data_ptr(), 300, hmap.ctypes.data, dt.data_ptr(), 300, 0)])
    arr, _, _keep = M.Context._wide_device_pairs([wide, bad], False)
    words = torch.zeros((8,), dtype=torch.int64, device=b.device)
    out = torch.empty((600, 4), dtype=torch.int32, device=b.device)
    p = M.Context._params(1, M.MODE_MUTUAL)
    w = lambda i: words[i:].data_ptr()
    h = C.c_void_p()
    b.use_torch_stream()
    assert b.ctx._L.b200m_plan_match_multiscale_batch(b.ctx._h, C.byref(p), arr, 2, src.shape[1] * 4, dim, 16, 40, None, None,
                                                      out.data_ptr(), 600, w(0), w(3), w(5), w(6), C.byref(h)) != 0
    assert not h.value
    assert b.ctx._L.b200m_last_error(b.ctx._h).decode() == \
        "b200m_plan_match_multiscale_batch: pair 1: scale 1: src_map is not device memory (host memory)"
    # a status word is required, and must be device memory too
    assert b.ctx._L.b200m_plan_match_multiscale_batch(b.ctx._h, C.byref(p), arr, 1, src.shape[1] * 4, dim, 16, 40, None, None,
                                                      out.data_ptr(), 600, w(0), w(3), w(5), None, C.byref(h)) != 0
    assert "null status" in b.ctx._L.b200m_last_error(b.ctx._h).decode()
    # no pair with source keypoints: only the finish step runs -- zero offsets and records, FLT_MAX averages, a clean status
    empty = torch.zeros((0, 4), dtype=torch.float32, device=b.device)
    no_rows = torch.zeros((0, src.shape[1]), dtype=torch.float32, device=b.device)
    pr = dict(src_scales=[(no_rows, None)], tgt_scales=[(dt, None)], src_kps_xyz=empty,
              tgt_kps_xyz=xyz, iss_radius_src=0.05, iss_radius_tgt=0.05)
    for gs in (False, True):
        pl = (b.plan_match_wide_local_batch(1, M.MODE_CLUSTER, [pr, pr], RADIUS, dim=dim) if gs else
              b.plan_match_wide_batch(1, M.MODE_CLUSTER, [pr, pr], dim=dim))
        g = _capture(torch, [pl])
        g.replay()
        got = pl.results()
        assert [r[0].shape[0] for r in got] == [0, 0]
        assert all(np.float32(r[1]) == np.float32(M.FLT_MAX) for r in got)
        assert int(pl.n_out.item()) == 0 and int(pl.status.item()) & MASK == MASK
        pl.close()
