"""Batches on a group (b200m_group_knn_batch / _match_batch / _match_multiscale_batch / _match_multiscale_local_batch,
Group.*_batch, match_many(devices=...)): the pairs split into contiguous ranges over the group's devices must give, byte for
byte, what the single-context batch form gives -- k-lists, records, offsets, averages, return code and error text.  Tests on
a group of one device run on any B200 box; tests on several devices skip on a one-GPU box."""
import ctypes
import dataclasses
import os
import subprocess

import numpy as np
import pytest

from lidar_global_registration_b200 import build as b200_build
from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth
from test_gpu_wide_batch import DTHR, GMODE, _case, _edge_cases, _matchers, _oracle
from test_gpu_wide_local import _guessed, _rigid, oracle_match_wide_local

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "group_batch_test")
RADIUS = 1.5


def _n_gpus():
    import torch
    return min(torch.cuda.device_count(), 8) if torch.cuda.is_available() else 0


@pytest.fixture(scope="module", autouse=True)
def _built():
    b200_build.build()
    M.load_library()


GROUPS = [[0], "split", [0, 1], "all"]


@pytest.fixture(scope="module", params=GROUPS, ids=["one", "one-split3", "two", "all"])
def group(request):
    """a group of one device, the same with three ranges per device (B200M_GROUP_RANGES: the split, the merge and the
    error selection across ranges run on a one-GPU box), two devices and every device"""
    n = _n_gpus()
    devs = list(range(n)) if request.param == "all" else [0] if request.param == "split" else request.param
    if len(devs) > n or (request.param == "all" and n <= 2):
        pytest.skip("needs %s GPUs" % ("more than two" if request.param == "all" else len(devs)))
    old = os.environ.get("B200M_GROUP_RANGES")
    if request.param == "split":
        os.environ["B200M_GROUP_RANGES"] = "3"   # read when the group is created
    try:
        g = M.Group(devs)
    finally:
        if old is None:
            os.environ.pop("B200M_GROUP_RANGES", None)
        else:
            os.environ["B200M_GROUP_RANGES"] = old
    with g:
        yield g


def _same_records(got, ref):
    assert len(got) == len(ref)
    for p, ((r, a), (e, ea)) in enumerate(zip(got, ref)):
        assert r.tobytes() == e.tobytes() and np.float32(a).tobytes() == np.float32(ea).tobytes(), p


def _same_lists(got, ref):
    assert len(got) == len(ref)
    for p, (g, e) in enumerate(zip(got, ref)):
        for a, b in zip(g, e):
            assert a.tobytes() == b.tobytes(), p


# ---- k-list and match batches --------------------------------------------------------------------------------------------
def _pairs(desc, sizes, seed, nan_frac=0.01):
    out = []
    for i, (ns, nt) in enumerate(sizes):
        s, t, dim = synth.make_pair(desc, max(ns, 1), max(nt, 1), seed=seed + i, nan_frac=nan_frac)
        out.append((s[:ns], t[:nt]))
    return out, dim


def _narrow_batches():
    """the batch-call test shapes, plus empty pairs, NaN rows, an aliased pair and one pair that dominates the cost"""
    odd, dim = _pairs("fpfh", [(700, 900), (0, 300), (255, 0), (256, 257), (1, 1), (3000, 2800), (400, 401)], 10)
    odd.append(odd[0])   # aliased: the same arrays twice
    nan = _pairs("shot", [(300, 310), (280, 290), (500, 200)], 30, nan_frac=0.3)
    return [("fpfh-odd", odd, dim), ("shot-nan", nan[0], nan[1])] + [
        ("fpfh-B%d" % b, _pairs("fpfh", [(200 + 37 * (i % 5), 230 + 23 * (i % 7)) for i in range(b)], 50)[0], 33) for b in (1, 2, 7, 64)]


NARROW = _narrow_batches()


@gpu
@pytest.mark.parametrize("name,pairs,dim", NARROW, ids=[n for n, _, _ in NARROW])
def test_knn_and_match_batch_equal_context(group, name, pairs, dim):
    with M.Context(0) as ctx:
        for k in (1, 2, 5):
            _same_lists(group.knn_batch(k, pairs, dim), ctx.knn_batch(k, pairs, dim))
        rng = np.random.default_rng(1)
        ts = [rng.random(len(s)).astype(np.float32) for s, _ in pairs]
        tt = [rng.random(len(t)).astype(np.float32) for _, t in pairs]
        for mode, k in ((M.MODE_ONE_SIDED, 1), (M.MODE_MUTUAL, 2), (M.MODE_RATIO, 2), (M.MODE_RATIO_MUTUAL, 3)):
            _same_records(group.match_batch(k, mode, pairs, dim), ctx.match_batch(k, mode, pairs, dim))
        _same_records(group.match_batch(2, M.MODE_MUTUAL, pairs, dim, distance_thr=0.7, thr_src=ts, thr_tgt=tt),
                      ctx.match_batch(2, M.MODE_MUTUAL, pairs, dim, distance_thr=0.7, thr_src=ts, thr_tgt=tt))


# ---- matcher-class batches ------------------------------------------------------------------------------------------------
def _wide_batches():
    ed = _edge_cases(2)
    ed[7][0]["src_scales"][1][0][:, :] = np.nan
    shot = [_case("shot", 2, 2, 200 + i, n_sk=300, n_tk=320) for i in range(3)]
    big = [_case("fpfh", 2, 1, 300, n_sk=2000, n_tk=2100)] + [_case("fpfh", 2, 1, 301 + i, n_sk=150, n_tk=160) for i in range(6)]
    out = [("edge", ed), ("shot", shot), ("dominant", big)]
    for b in (1, 2, 7, 64):
        out.append(("B%d" % b, [_case("fpfh", 2, 1 + i % 2, 400 + i, n_sk=150 + 13 * (i % 4), n_tk=170) for i in range(b)]))
    out.append(("aliased", [out[1][1][0], out[1][1][1], out[1][1][0]]))
    return out


WIDE = _wide_batches()


def _wide_args(cases):
    return [c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], cases[0][3]


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
@pytest.mark.parametrize("name,cases", WIDE, ids=[n for n, _ in WIDE])
def test_wide_batch_equals_context(group, name, cases, mode):
    pairs, ts, tt, dim = _wide_args(cases)
    with M.Context(0) as ctx:
        ref = ctx.match_wide_batch(2, GMODE[mode], pairs, dim, 40, DTHR, ts, tt)
        _same_records(group.match_wide_batch(2, GMODE[mode], pairs, dim, 40, DTHR, ts, tt), ref)
        _same_records(group.match_wide_batch(2, GMODE[mode], pairs, dim, 40, DTHR),
                      ctx.match_wide_batch(2, GMODE[mode], pairs, dim, 40, DTHR))
    if name == "B7":   # and the oracle's composition
        for p, (r, a) in enumerate(ref):
            if len(pairs[p]["src_kps_xyz"]) and len(pairs[p]["tgt_kps_xyz"]) and pairs[p]["src_scales"]:
                e, ea = _oracle(mode, 2, pairs[p], ts[p], tt[p])
                assert r.tobytes() == e.tobytes() and a == ea


@gpu
@pytest.mark.parametrize("mode", ["one_sided", "mutual", "cluster"])
@pytest.mark.parametrize("name,cases", [w for w in WIDE if w[0] in ("edge", "dominant", "B2", "B7", "B64")],
                         ids=["edge", "dominant", "B2", "B7", "B64"])
def test_wide_local_batch_equals_context(group, name, cases, mode):
    pairs, ts, tt, dim = _wide_args(cases)
    pairs = [_guessed(pr, _rigid(i)) for i, pr in enumerate(pairs)]
    with M.Context(0) as ctx:
        ref = ctx.match_wide_local_batch(2, GMODE[mode], pairs, RADIUS, dim, 40, DTHR, ts, tt)
    _same_records(group.match_wide_local_batch(2, GMODE[mode], pairs, RADIUS, dim, 40, DTHR, ts, tt), ref)
    if name == "B7":
        for p, (r, a) in enumerate(ref):
            if len(pairs[p]["src_kps_xyz"]) and len(pairs[p]["tgt_kps_xyz"]) and pairs[p]["src_scales"]:
                e, ea = oracle_match_wide_local(mode, pairs[p], 2, RADIUS, thr_q=ts[p], thr_t=tt[p])
                assert r.tobytes() == e.tobytes() and a == ea


# ---- errors --------------------------------------------------------------------------------------------------------------
def _raw(target, fn, *a):
    """(return code, error text) of a direct C call on a Context or a Group"""
    is_group = isinstance(target, M.Group)
    L = target._L
    rc = getattr(L, ("b200m_group_" if is_group else "b200m_") + fn)(target._h, *a)
    err = (L.b200m_group_last_error(target._h) if is_group else L.b200m_last_error(target._h)).decode() if rc else ""
    return rc, err


def _match_batch_raw(target, pairs, dim, cap, mode=M.MODE_MUTUAL, k=2):
    keep, arr, stride, ns = M.Context._pairs(pairs, dim)
    out = np.zeros(max(cap, 1), M.CORR_DTYPE)
    offsets = np.full(len(pairs) + 1, 77, np.uint64)
    avg = np.zeros(max(len(pairs), 1), np.float32)
    p = M.Context._params(k, mode)
    rc, err = _raw(target, "match_batch", ctypes.byref(p), arr, len(pairs), stride, dim, None, None, out.ctypes.data, cap,
                   offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), avg.ctypes.data)
    return rc, err, offsets, avg, out


def _wide_raw(target, pairs, dim, cap, mode=M.MODE_MUTUAL, k=2):
    """b200m_match_multiscale_batch with a given cap through the Python marshalling, with its outputs"""
    box = {}

    class Spy:
        def __init__(self, L):
            self.L = L

        def __getattr__(self, name):
            f = getattr(self.L, name)
            if not name.endswith("match_multiscale_batch"):
                return f

            def call(*a):
                a = list(a)
                a[11] = cap
                box["rc"] = f(*a)
                box["offsets"] = np.ctypeslib.as_array(a[12], shape=(len(pairs) + 1,)).copy()
                box["avg"] = np.ctypeslib.as_array(ctypes.cast(a[13], ctypes.POINTER(ctypes.c_float)), shape=(len(pairs),)).copy()
                return box["rc"]
            return call

    L = target._L
    target._L = Spy(L)
    try:
        target.match_wide_batch(k, mode, pairs, dim)
        err = ""
    except M.B200MatchError as e:
        err = str(e)
    finally:
        target._L = L
    return box.get("rc", 1), err, box.get("offsets"), box.get("avg")


def _bad_map(pr, scale, entry, value):
    pr = dict(pr)
    sc = list(pr["src_scales"])
    m = np.arange(len(sc[scale][0]), dtype=np.int32) if sc[scale][1] is None else sc[scale][1].copy()
    m[entry] = value
    sc[scale] = (sc[scale][0], m)
    pr["src_scales"] = sc
    return pr


@gpu
def test_errors_equal_context(group):
    cases = [_case("fpfh", 2, 2, 500 + i, n_sk=300, n_tk=320) for i in range(4)]   # equal costs: ranges of equal length
    pairs, _, _, dim = _wide_args(cases)
    with M.Context(0) as ctx:
        def same(fn):
            e = fn(ctx)
            g = fn(group)
            assert e[0] != 0 and g[0] != 0
            assert g[1] == e[1]
            return e[1]

        def wide(ps, mode=M.MODE_MUTUAL):
            def f(t):
                try:
                    t.match_wide_batch(2, mode, ps, dim)
                    return 0, ""
                except M.B200MatchError as e:
                    return 1, str(e)
            return f

        # a bad map in a later pair and scale (device 0 of two) and one in an earlier scale of a later pair (device 1): the
        # smallest (scale, pair, side) is the single form's
        bad = list(pairs)
        bad[1] = _bad_map(bad[1], 1, 5, 10 ** 6)
        bad[3] = _bad_map(bad[3], 0, 7, -3)
        assert same(wide(bad)).endswith("pair 3, scale 0: an index map entry of the source cloud is outside its keypoint range")
        bad[3] = pairs[3]
        assert "pair 1, scale 1:" in same(wide(bad))
        # a check that fails in pairs of both devices: the lowest pair; and a check failure wins over a bad map
        nox = [dict(p) for p in pairs]
        for i in (1, 3):
            nox[i]["n_src_kps"] = len(nox[i]["src_kps_xyz"])
            nox[i]["src_kps_xyz"] = None
        assert same(wide(nox, M.MODE_CLUSTER)).endswith("pair 1: null keypoint coordinates")
        nox[0] = _bad_map(pairs[0], 0, 0, 10 ** 6)
        nox[1] = pairs[1]
        assert same(wide(nox, M.MODE_CLUSTER)).endswith("pair 3: null keypoint coordinates")
        deep = [dict(p) for p in pairs]
        deep[2]["src_scales"] = deep[2]["src_scales"] * 3
        deep[2]["tgt_scales"] = deep[2]["tgt_scales"] * 3
        assert "pair 2: n_scales * k > 128" in same(lambda t: _try(lambda: t.match_wide_batch(32, M.MODE_MUTUAL, deep, dim)))
        # params the single form rejects, and an empty batch
        assert "mode must be ONE_SIDED, MUTUAL or CLUSTER" in same(wide(pairs, M.MODE_RATIO))
        assert "params.k" in same(lambda t: _try(lambda: t.match_batch(0, M.MODE_MUTUAL, [(pairs[0]["src_scales"][0][0],) * 2], dim)))
        assert group.match_wide_batch(2, M.MODE_MUTUAL, [], dim) == [] and group.knn_batch(2, [], dim) == []
        # a null descriptor pointer names the batch's pair
        narrow, ndim = _pairs("fpfh", [(300, 310)] * 4, 70)
        keep, arr, stride, _ = M.Context._pairs(narrow, ndim)
        arr[3].src = None
        p = M.Context._params(2, M.MODE_KNN_ONLY)
        out = [np.zeros((1200, 2), np.int32), np.zeros((1200, 2), np.float32), np.zeros(1200, np.int32)]
        e = _raw(ctx, "knn_batch", ctypes.byref(p), arr, 4, stride, ndim, *[o.ctypes.data for o in out])
        g = _raw(group, "knn_batch", ctypes.byref(p), arr, 4, stride, ndim, *[o.ctypes.data for o in out])
        assert e[0] and g == e and e[1].endswith("null descriptor pointer in pair 3")
        # after an error the offsets are the single form's (zeroed once the arguments passed)
        offs = []
        for target in (ctx, group):
            o = np.full(5, 77, np.uint64)
            rc = _raw(target, "match_batch", ctypes.byref(M.Context._params(2, M.MODE_MUTUAL)), arr, 4, stride, ndim, None, None,
                      np.zeros(8, M.CORR_DTYPE).ctypes.data, 8, o.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), None)
            assert rc[0] and rc[1].endswith("null descriptor pointer in pair 3")
            offs.append(o)
        assert offs[0].tobytes() == offs[1].tobytes() and not offs[0].any()
        bad = list(pairs)
        bad[1] = _bad_map(bad[1], 1, 5, 10 ** 6)
        e, g = _wide_raw(ctx, bad, dim, 10 ** 6), _wide_raw(group, bad, dim, 10 ** 6)
        assert e[0] and g[0] and g[1] == e[1] and g[2].tobytes() == e[2].tobytes() and not e[2].any()
        # cap too small: same error, offsets and averages still filled
        for cap in (0, 1, 5):
            e = _match_batch_raw(ctx, narrow, ndim, cap)
            g = _match_batch_raw(group, narrow, ndim, cap)
            assert e[0] and g[0] and g[1] == e[1] and "capacity too small" in e[1]
            assert g[2].tobytes() == e[2].tobytes() and g[3].tobytes() == e[3].tobytes() and e[2][-1] > 5
            e = _wide_raw(ctx, pairs, dim, cap)
            g = _wide_raw(group, pairs, dim, cap)
            assert e[0] and g[0] and g[1] == e[1] and "capacity too small" in e[1]
            assert g[2].tobytes() == e[2].tobytes() and g[3].tobytes() == e[3].tobytes()


def _try(f):
    try:
        f()
        return 0, ""
    except M.B200MatchError as e:
        return 1, str(e)


def test_null_group_fails_with_the_single_form_text():
    L = M.load_library()
    p = M.Context._params(2, M.MODE_MUTUAL)
    assert L.b200m_group_knn_batch(None, ctypes.byref(p), None, 0, 132, 33, None, None, None) != 0
    assert L.b200m_group_last_error(None).decode() == "null context"


# ---- match_many on devices ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("cls_id,k,n_scales,coords", [(M.MATCHING_CLUSTER, 2, 2, True), (M.MATCHING_LEFT_TO_RIGHT, 2, 1, True),
                                                      (M.MATCHING_ONE_SIDED, 1, 1, False)], ids=["cluster", "lr", "narrow"])
@pytest.mark.parametrize("guessed", [False, True], ids=["unguessed", "guessed"])
def test_match_many_on_devices_equals_match_many(cls_id, k, n_scales, coords, guessed):
    if guessed and not coords:
        pytest.skip("a guess needs keypoint coordinates")
    makers = _matchers(cls_id, k, n_scales, [610, 611, 612, 613, 614], coords)

    def make():
        ms = [mk() for mk in makers]
        if guessed:
            for i, m in enumerate(ms):
                m.parameters = dataclasses.replace(m.parameters, guess=_rigid(i), match_search_radius=RADIUS)
        return ms

    ref_ms = make()
    ref = M.match_many(ref_ms)
    n = _n_gpus()
    for devs in ([0], list(range(n))) if n > 1 else ([0],):
        ms = make()
        got = M.match_many(ms, devices=devs)
        for a, b, ma, mb in zip(got, ref, ms, ref_ms):
            assert a.tobytes() == b.tobytes() and ma.get_average_distance() == mb.get_average_distance()
    assert sum(len(r) for r in ref) > 0


# ---- the C++ shim's matchMany on several devices --------------------------------------------------------------------------
def _build_exe():
    b200_build.build()
    src = os.path.join(ROOT, "tests", "cpp", "group_batch_test.cpp")
    deps = [src, os.path.join(ROOT, "include", "b200match_shim.hpp"), os.path.join(ROOT, "include", "b200match.h")]
    if os.path.exists(EXE) and all(os.path.getmtime(EXE) >= os.path.getmtime(d) for d in deps):
        return EXE
    libdir = os.path.join(ROOT, "lidar_global_registration_b200")
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", EXE,
                    "-L", libdir, "-l:libb200match.so", "-Wl,-rpath," + libdir], check=True)
    return EXE


def test_group_batch_program_compiles_and_links():
    r = subprocess.run([_build_exe()], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr


@gpu
def test_cpp_match_many_on_devices_equals_one_device():
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    r = subprocess.run([_build_exe(), str(n)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("devices {0} ==") == 6


@gpu
def test_group_knn_and_match_refuse_after_a_batch_until_uploaded_again():
    """a batch leaves every device with its own range's sets: the whole-problem calls must not size their outputs from
    the sets uploaded before"""
    pairs, dim = _pairs("fpfh", [(300, 310), (500, 290)], 80)
    s, t, _ = synth.make_pair("fpfh", 700, 650, seed=81)
    with M.Group([0]) as g, M.Context(0) as ctx:
        g.upload(0, s, dim)
        g.upload(1, t, dim)
        g.knn_batch(2, pairs, dim)
        with pytest.raises(M.B200MatchError, match="upload both sides again"):
            g.knn(2)
        with pytest.raises(M.B200MatchError, match="upload both sides again"):
            g.match(2, M.MODE_MUTUAL)
        with pytest.raises(M.B200MatchError):   # a failed batch replaces the sets too
            g.match_wide_batch(2, M.MODE_RATIO, [_case("fpfh", 2, 1, 82, n_sk=100, n_tk=120)[0]], dim)
        g.upload(0, s, dim)
        with pytest.raises(M.B200MatchError, match="upload both sides again"):
            g.knn(2)
        g.upload(1, t, dim)
        ctx.upload(0, s, dim)
        ctx.upload(1, t, dim)
        for a, b in zip(g.knn(2), ctx.knn(2)):
            assert a.tobytes() == b.tobytes()
