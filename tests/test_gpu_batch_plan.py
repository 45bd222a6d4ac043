"""Batch plans (b200m_plan_knn_batch / b200m_plan_match_batch / b200m_plan_run through GpuBackend.plan_*): a plan is bound
once and its run only enqueues, so it is captured in torch.cuda.graph (global capture mode: a sync, an allocation or a
pageable copy inside run would fail the capture).  After every input tensor is rewritten in place, a replay must give, byte
for byte, what the device form (GpuBackend.knn_batch / match_batch) gives on the new data -- inside and outside the
certificate's window, with a capacity below the records found, and after the caller's own context has grown its
workspaces.  GPU tests run with -m gpu on a B200; the C-ABI surface is checked without one."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLAN_ENTRIES = ["b200m_plan_knn_batch", "b200m_plan_match_batch", "b200m_plan_run", "b200m_plan_destroy",
                "b200m_plan_last_error"]
MODES = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "ratio": M.MODE_RATIO, "ratio_mutual": M.MODE_RATIO_MUTUAL}
DTHR = np.float32(0.7)
# empty sides, one row, the 255 / 256 / 257-row edges of a tile; pair 7 aliases pair 6's source set on both sides
SIZES = [(0, 40), (1, 1), (255, 257), (256, 256), (257, 255), (40, 0), (700, 650)]


def _lib_built():
    return os.path.exists(M._LIB_PATH)


# ---- C-ABI surface (no GPU) -----------------------------------------------------------------------------------------------
def test_plan_entries_exported_and_declared():
    text = open(os.path.join(ROOT, "include", "b200match.h")).read()
    declared = set(re.findall(r"B200M_API\s+[\w\s\*]+?\b(b200m_\w+)\s*\(", text))
    for name in PLAN_ENTRIES:
        assert name in M.EXPORTS, name
        assert name in declared, name


def test_plan_entries_have_argtypes():
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    for name in PLAN_ENTRIES:
        assert getattr(L, name).argtypes is not None, name
    assert len(L.b200m_plan_knn_batch.argtypes) == 10
    assert len(L.b200m_plan_match_batch.argtypes) == 14
    assert L.b200m_plan_destroy.restype is None
    assert L.b200m_plan_last_error.restype is C.c_char_p


def test_plan_without_context_fails_loudly():
    """no context (as without a device: b200m_create fails first, there is no CPU fallback) -> an error, no plan"""
    if not _lib_built():
        pytest.skip("library not built")
    L = M.load_library()
    p = M.Context._params(1, M.MODE_MUTUAL)
    pairs = M.Context._device_pairs([(0, 0, 0, 0)])
    h = C.c_void_p(1234)
    assert L.b200m_plan_knn_batch(None, C.byref(p), pairs, 1, 132, 33, None, None, None, C.byref(h)) != 0
    assert not h.value
    assert L.b200m_plan_last_error(None).decode() == "null context"
    h = C.c_void_p(1234)
    assert L.b200m_plan_match_batch(None, C.byref(p), pairs, 1, 132, 33, None, None, None, 0, None, None, None,
                                    C.byref(h)) != 0
    assert not h.value
    assert L.b200m_plan_run(None, None) != 0
    L.b200m_plan_destroy(None)


def test_plan_without_device_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(M.B200MatchError):
        M.Context(0)


# ---- fixtures and helpers (GPU) -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def backend():
    from lidar_global_registration_b200 import device as D
    b = D.GpuBackend(0)
    yield b
    b.close()


def _host_sets(desc, sizes, seed):
    out = []
    for i, (ns, nt) in enumerate(sizes):
        s, t, dim = synth.make_pair(desc, max(ns, 1), max(nt, 1), seed=seed * 100 + i, nan_frac=0.02)
        out.append((np.ascontiguousarray(s[:ns]), np.ascontiguousarray(t[:nt])))
    return out, synth.DESCRIPTORS[desc][0]


class Bound:
    """One device tensor per side holding every set as a row slice (3 junk rows between sets), an extra pair that aliases
    the last pair's source set on both sides (unless alias is False), and threshold tensors split per pair.  write() rewrites them in place."""

    def __init__(self, dev, host_pairs, alias=True):
        import torch
        self.torch = torch
        self.sizes = [(s.shape[0], t.shape[0]) for s, t in host_pairs]
        width = host_pairs[0][0].shape[1]
        self.offs, self.big = [], []
        for side in (0, 1):
            offs, o = [], 0
            for n in (sz[side] for sz in self.sizes):
                offs.append(o)
                o += n + 3
            self.offs.append(offs)
            self.big.append(torch.zeros((o, width), dtype=torch.float32, device=dev))
        self.pairs = [(self.big[0][a:a + ns], self.big[1][b:b + nt])
                      for a, b, (ns, nt) in zip(self.offs[0], self.offs[1], self.sizes)]
        if alias:
            last = self.pairs[-1][0]
            self.pairs.append((last, last))
        counts = [(p[0].shape[0], p[1].shape[0]) for p in self.pairs]
        self.thr_all = [torch.zeros((sum(c[s] for c in counts),), dtype=torch.float32, device=dev) for s in (0, 1)]
        self.thr = [list(self.thr_all[s].split([c[s] for c in counts])) for s in (0, 1)]
        self.write(host_pairs, 0)

    def write(self, host_pairs, seed):
        torch = self.torch
        for side in (0, 1):
            for o, pr in zip(self.offs[side], host_pairs):
                a = pr[side]
                self.big[side][o:o + a.shape[0]].copy_(torch.from_numpy(a))
            self.thr_all[side].copy_(torch.from_numpy(np.random.default_rng(seed + side).random(self.thr_all[side].shape[0])
                                                      .astype(np.float32)))


def _capture(torch, plans):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for p in plans:
            p.run()
    return g


def _same_lists(plan, ref):
    got = plan.results()
    assert len(got) == len(ref)
    for p, (g, r) in enumerate(zip(got, ref)):
        for x, y in zip(g, r):
            assert x.cpu().numpy().tobytes() == y.cpu().numpy().tobytes(), "pair %d" % p


def _same_records(plan, ref):
    got = plan.results()
    assert len(got) == len(ref)
    for p, ((recs, avg), (rrecs, ravg)) in enumerate(zip(got, ref)):
        assert recs.cpu().numpy().tobytes() == rrecs.cpu().numpy().tobytes(), "pair %d records" % p
        assert np.float32(avg).tobytes() == np.float32(ravg).tobytes(), "pair %d average" % p
    n = sum(r[0].shape[0] for r in ref)
    assert int(plan.n_out.item()) == n
    offs = np.cumsum([0] + [r[0].shape[0] for r in ref])
    assert plan.offsets.cpu().numpy().tolist() == offs.tolist()


# ---- capture and replay ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [1, 2, 5])
@pytest.mark.parametrize("desc", ["fpfh", "rops", "shot", "usc"])
def test_capture_and_replay_equals_device_form(backend, desc, k):
    import torch
    b = backend
    first, dim = _host_sets(desc, SIZES, 1)
    bd = Bound(b.device, first)
    modes = [m for m in MODES if k >= 2 or "ratio" not in m]
    plans = [b.plan_knn_batch(k, bd.pairs, dim)]
    for m in modes:
        plans.append(b.plan_match_batch(k, MODES[m], bd.pairs, dim, distance_thr=DTHR))
        plans.append(b.plan_match_batch(k, MODES[m], bd.pairs, dim, distance_thr=DTHR, thr_src=bd.thr[0], thr_tgt=bd.thr[1]))
    g = _capture(torch, plans)
    for seed in (2, 3):
        new, _ = _host_sets(desc, SIZES, seed)
        bd.write(new, seed)
        g.replay()
        _same_lists(plans[0], b.knn_batch(k, bd.pairs, dim))
        i = 1
        for m in modes:
            for thr in (False, True):
                kw = dict(thr_src=bd.thr[0], thr_tgt=bd.thr[1]) if thr else {}
                _same_records(plans[i], b.match_batch(k, MODES[m], bd.pairs, dim, distance_thr=DTHR, **kw))
                i += 1
    for p in plans:
        p.close()


# ---- routing on the device ------------------------------------------------------------------------------------------------
def _route(b, pairs, dim):
    """candidate launches of a device-form call on this data: > 0 iff it ran on the tensor cores"""
    b.ctx.set_profiling(True)
    b.ctx.reset_stats()
    b.knn_batch(2, pairs, dim)
    launches = b.ctx.stats()["candidate_launches"]
    b.ctx.set_profiling(False)
    return launches > 0


@gpu
@pytest.mark.parametrize("dim", [33, 352, 1960])
def test_replay_routes_on_the_device(backend, dim):
    """replays whose data leaves the certificate's window (one pair at 1e20, subnormals, one float beyond either edge) answer
    as the device form's exact path; in-window replays (the last float inside either edge, ordinary data) as its tensor-core
    path -- the plan takes the route the host would have taken, without the host"""
    import torch
    import test_gpu_magnitudes as TM
    b = backend
    rng = np.random.default_rng(dim)
    sizes = [300, 260]

    def ordinary(scale=1.0):
        return [((rng.random((n, dim)) * scale).astype(np.float32), (rng.random((n, dim)) * scale).astype(np.float32))
                for n in sizes]

    def symmetric(edge):
        return [TM._symmetric(rng, n, dim, edge, TM._unit(edge)) for n in sizes]

    hi, lo = TM.upper_edge(dim), TM.lower_edge(dim)
    big = ordinary()
    big[0] = (big[0][0] * np.float32(1e20), big[0][1] * np.float32(1e20))
    cases = [("1e20", big, False), ("subnormal", ordinary(1e-40), False), ("hi_in", symmetric(hi), True),
             ("hi_out", symmetric(TM._outside(hi, True)), False), ("lo_in", symmetric(lo), True),
             ("lo_out", symmetric(TM._outside(lo, False)), False), ("ordinary", ordinary(), True)]
    bd = Bound(b.device, ordinary(), alias=False)   # every pair symmetric: the batch's centre stays exactly 0
    pk = b.plan_knn_batch(2, bd.pairs, dim)
    pm = b.plan_match_batch(2, M.MODE_MUTUAL, bd.pairs, dim)
    g = _capture(torch, [pk, pm])
    for seed, (name, data, inside) in enumerate(cases):
        bd.write(data, seed)
        g.replay()
        _same_lists(pk, b.knn_batch(2, bd.pairs, dim))
        _same_records(pm, b.match_batch(2, M.MODE_MUTUAL, bd.pairs, dim))
        assert _route(b, bd.pairs, dim) == inside, name
    pk.close()
    pm.close()


# ---- capacity -------------------------------------------------------------------------------------------------------------
@gpu
def test_capacity_is_reported_not_enforced(backend):
    import torch
    b = backend
    data, dim = _host_sets("fpfh", SIZES, 7)
    bd = Bound(b.device, data)
    ref = b.match_batch(2, M.MODE_MUTUAL, bd.pairs, dim)
    n = sum(r[0].shape[0] for r in ref)
    assert n > 10
    cap = n // 3
    sentinel = -7
    out = torch.full((n + 100, 4), sentinel, dtype=torch.int32, device=b.device)
    offsets = torch.zeros((len(bd.pairs) + 1,), dtype=torch.int64, device=b.device)
    avg = torch.zeros((len(bd.pairs),), dtype=torch.float32, device=b.device)
    n_out = torch.zeros((1,), dtype=torch.int64, device=b.device)
    ptrs, stride = b._set_pairs(bd.pairs, dim)
    p = M.Context._params(2, M.MODE_MUTUAL)
    arr = M.Context._device_pairs(ptrs)
    L, h = b.ctx._L, C.c_void_p()
    b.use_torch_stream()
    assert L.b200m_plan_match_batch(b.ctx._h, C.byref(p), arr, len(ptrs), stride, dim, None, None, out.data_ptr(), cap,
                                    offsets.data_ptr(), avg.data_ptr(), n_out.data_ptr(), C.byref(h)) == 0, \
        L.b200m_last_error(b.ctx._h).decode()
    try:
        out[:cap].fill_(sentinel)
        n_out.zero_()
        assert L.b200m_plan_run(h, C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        torch.cuda.synchronize()
        assert int(n_out.item()) == n
        full = torch.cat([r[0] for r in ref])
        assert out[:cap].cpu().numpy().tobytes() == full[:cap].cpu().numpy().tobytes()
        assert bool((out[cap:] == sentinel).all())
        assert offsets.cpu().numpy().tolist() == np.cumsum([0] + [r[0].shape[0] for r in ref]).tolist()
        assert avg.cpu().numpy().tobytes() == np.array([r[1] for r in ref], np.float32).tobytes()
    finally:
        L.b200m_plan_destroy(h)


@gpu
def test_refusals_and_empty_batches(backend):
    b = backend
    data, dim = _host_sets("fpfh", [(50, 60)], 8)
    host = data[0][0]
    with pytest.raises(M.B200MatchError, match="not device memory"):
        bad = M.Context._device_pairs([(host.ctypes.data, 50, host.ctypes.data, 50)])
        p = M.Context._params(1, M.MODE_MUTUAL)
        h = C.c_void_p()
        b.ctx._ck(b.ctx._L.b200m_plan_knn_batch(b.ctx._h, C.byref(p), bad, 1, 132, dim, None, None, None, C.byref(h)))
    import torch
    empty = torch.zeros((0, dim), dtype=torch.float32, device=b.device)
    other = torch.ones((5, dim), dtype=torch.float32, device=b.device)
    pm = b.plan_match_batch(1, M.MODE_MUTUAL, [(empty, other)], dim)
    pk = b.plan_knn_batch(1, [(empty, other)], dim)
    g = _capture(torch, [pm, pk])
    g.replay()
    got = pm.results()
    assert len(got) == 1 and got[0][0].shape[0] == 0 and np.float32(got[0][1]) == np.float32(M.FLT_MAX)
    assert int(pm.n_out.item()) == 0
    pm.close()
    pk.close()


# ---- ownership ------------------------------------------------------------------------------------------------------------
@gpu
def test_caller_context_growth_does_not_move_the_plan(backend):
    import torch
    b = backend
    data, dim = _host_sets("shot", SIZES, 11)
    bd = Bound(b.device, data)
    pk = b.plan_knn_batch(2, bd.pairs, dim)
    pm = b.plan_match_batch(2, M.MODE_MUTUAL, bd.pairs, dim)
    g = _capture(torch, [pk, pm])
    large, _ = _host_sets("shot", [(3000, 3500), (2600, 2900), (4000, 1000)], 12)
    lb = Bound(b.device, large)
    b.match_batch(2, M.MODE_MUTUAL, lb.pairs, dim)
    b.knn_batch(5, lb.pairs, dim)
    new, _ = _host_sets("shot", SIZES, 13)
    bd.write(new, 13)
    g.replay()
    _same_lists(pk, b.knn_batch(2, bd.pairs, dim))
    _same_records(pm, b.match_batch(2, M.MODE_MUTUAL, bd.pairs, dim))
    pk.close()
    pm.close()
