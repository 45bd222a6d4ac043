"""The device-resident batch calls (b200m_knn_batch_device, b200m_match_batch_device, b200m_match_multiscale_batch_device,
b200m_match_multiscale_local_batch_device through GpuBackend and Context): on the same seeded data every pair's k-lists,
records, offsets and averages must equal, byte for byte, what the host forms (Context.knn_batch / match_batch /
match_wide_batch / match_wide_local_batch) return.  The internals must be the same too (FP16 operand tiles, candidate
counts), launches per call must not grow with the number of pairs, and host pointers are refused before anything is
launched.  GPU tests run with -m gpu on a B200; the argument layout is checked without one."""
import ctypes

import numpy as np
import pytest

from lidar_global_registration_b200 import matcher as M
from lidar_global_registration_b200 import synth

gpu = pytest.mark.gpu
DTHR = np.float32(0.7)
MODES = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "ratio": M.MODE_RATIO, "ratio_mutual": M.MODE_RATIO_MUTUAL}
WMODES = {"one_sided": M.MODE_ONE_SIDED, "mutual": M.MODE_MUTUAL, "cluster": M.MODE_CLUSTER}
DEVICE_ENTRIES = ["b200m_knn_batch_device", "b200m_match_batch_device", "b200m_match_multiscale_batch_device",
                  "b200m_match_multiscale_local_batch_device"]


def test_device_entries_exported_and_declared():
    for name in DEVICE_ENTRIES:
        assert name in M.EXPORTS
        host = name[:-len("_device")]
        assert host in M.EXPORTS


def test_device_entries_take_host_form_arguments():
    L = M.load_library() if _lib_built() else None
    if L is None:
        pytest.skip("library not built")
    for name in DEVICE_ENTRIES:
        assert getattr(L, name).argtypes == getattr(L, name[:-len("_device")]).argtypes


def _lib_built():
    import os
    return os.path.exists(M._LIB_PATH)


# ---- helpers -----------------------------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


def _backend():
    from lidar_global_registration_b200 import device as D
    return D.GpuBackend(0)


def _sets(desc, sizes, seed):
    """[(src, tgt)] float32 AoS host arrays (the descriptor type's full row, SHOT: 361 floats) and dim"""
    out, dim = [], None
    for i, (ns, nt) in enumerate(sizes):
        s, t, dim = synth.make_pair(desc, max(ns, 1), max(nt, 1), seed=seed * 100 + i, nan_frac=0.02)
        out.append((np.ascontiguousarray(s[:ns]), np.ascontiguousarray(t[:nt])))
    return out, dim


def _as_slices(pairs, dev):
    """every set as a row slice of ONE device tensor per side (gaps of 3 rows between sets)"""
    torch = _torch()
    width = pairs[0][0].shape[1]
    res = []
    for side in (0, 1):
        blocks, offs, o = [], [], 0
        for pr in pairs:
            blocks += [pr[side], np.full((3, width), 7.0, np.float32)]
            offs.append(o)
            o += pr[side].shape[0] + 3
        big = torch.from_numpy(np.concatenate(blocks)).to(dev)
        res.append([big[a:a + pr[side].shape[0]] for a, pr in zip(offs, pairs)])
    return list(zip(res[0], res[1]))


def _same_lists(got, ref):
    assert len(got) == len(ref)
    for (gi, gd, gc), (ri, rd, rc) in zip(got, ref):
        assert gi.cpu().numpy().tobytes() == ri.tobytes()
        assert gd.cpu().numpy().tobytes() == rd.tobytes()
        assert gc.cpu().numpy().tobytes() == rc.tobytes()


def _same_records(got, ref):
    assert len(got) == len(ref)
    for p, ((recs, avg), (rrecs, ravg)) in enumerate(zip(got, ref)):
        assert recs.cpu().numpy().view(M.CORR_DTYPE).reshape(-1).tobytes() == rrecs.tobytes(), "pair %d records" % p
        assert np.float32(avg).tobytes() == np.float32(ravg).tobytes(), "pair %d average" % p


SIZES = [(0, 40), (1, 1), (255, 257), (256, 256), (257, 255), (40, 0), (700, 650)]


# ---- k-list seam ----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("desc,k", [("fpfh", 1), ("fpfh", 5), ("rops", 2), ("shot", 2), ("shot", 5)])
def test_knn_batch_device_equals_host(desc, k):
    pairs, dim = _sets(desc, SIZES, 1)
    with M.Context(0) as ctx:
        ref = ctx.knn_batch(k, pairs, dim)
    b = _backend()
    got = b.knn_batch(k, _as_slices(pairs, b.device), dim)
    _same_lists(got, ref)
    b.close()


@gpu
@pytest.mark.parametrize("desc", ["fpfh", "rops", "shot"])
@pytest.mark.parametrize("mode", list(MODES))
def test_match_batch_device_equals_host(desc, mode):
    torch = _torch()
    k = 2 if "ratio" in mode else {"fpfh": 1, "rops": 2, "shot": 5}[desc]
    pairs, dim = _sets(desc, SIZES, 2)
    rng = np.random.default_rng(3)
    ts = [rng.random(len(s)).astype(np.float32) for s, _ in pairs]
    tt = [rng.random(len(t)).astype(np.float32) for _, t in pairs]
    b = _backend()
    for thr in (False, True):
        with M.Context(0) as ctx:
            ref = ctx.match_batch(k, MODES[mode], pairs, dim, distance_thr=DTHR, thr_src=ts if thr else None,
                                  thr_tgt=tt if thr else None)
        dts = [torch.from_numpy(a).to(b.device) for a in ts] if thr else None
        dtt = [torch.from_numpy(a).to(b.device) for a in tt] if thr else None
        got = b.match_batch(k, MODES[mode], _as_slices(pairs, b.device), dim, distance_thr=DTHR, thr_src=dts, thr_tgt=dtt)
        _same_records(got, ref)
    b.close()


@gpu
def test_aliased_sets_and_empty_batch():
    torch = _torch()
    src, tgt, dim = synth.make_pair("fpfh", 3000, 2000, seed=5, nan_frac=0.02)
    subs = [tgt[a:a + 500] for a in range(0, 2000, 500)]
    host_pairs = [(src, t) for t in subs] + [(src, src)]
    b = _backend()
    ds, dt = torch.from_numpy(src).to(b.device), torch.from_numpy(tgt).to(b.device)
    dev_pairs = [(ds, dt[a:a + 500]) for a in range(0, 2000, 500)] + [(ds, ds)]
    with M.Context(0) as ctx:
        ref = ctx.match_batch(1, M.MODE_MUTUAL, host_pairs, dim)
        refk = ctx.knn_batch(2, host_pairs, dim)
        assert ctx.match_batch(1, M.MODE_MUTUAL, [], dim) == []
    _same_records(b.match_batch(1, M.MODE_MUTUAL, dev_pairs, dim), ref)
    _same_lists(b.knn_batch(2, dev_pairs, dim), refk)
    assert b.match_batch(1, M.MODE_MUTUAL, [], dim) == []
    assert b.knn_batch(1, [], dim) == []
    assert b.match_wide_batch(1, M.MODE_MUTUAL, [], dim) == []
    b.close()


@gpu
def test_same_internals_as_host_form():
    """the segmented pack gives the staging path's FP16 tiles (same centre and scale) and the same candidate counts"""
    pairs, dim = _sets("fpfh", SIZES, 4)
    b = _backend()
    dev_pairs = _as_slices(pairs, b.device)
    for call in ("knn", "match"):
        with M.Context(0) as ctx:
            ctx.set_profiling(True)
            ctx.reset_stats()
            if call == "knn":
                ctx.knn_batch(2, pairs, dim)
            else:
                ctx.match_batch(2, M.MODE_MUTUAL, pairs, dim)
            hs = ctx.stats()
            hops = [ctx.debug_operands(s, q) for s in (0, 1) for q in (0, 1)]
        b.ctx.set_profiling(True)
        b.ctx.reset_stats()
        if call == "knn":
            b.knn_batch(2, dev_pairs, dim)
        else:
            b.match_batch(2, M.MODE_MUTUAL, dev_pairs, dim)
        ds = b.ctx.stats()
        dops = [b.ctx.debug_operands(s, q) for s in (0, 1) for q in (0, 1)]
        for h, d in zip(hops, dops):
            for x, y in zip(h, d):
                assert np.asarray(x).tobytes() == np.asarray(y).tobytes()
        for key in ("rows_total", "candidates", "rows_flagged", "pairs_scored"):
            assert hs[key] == ds[key], key
    b.close()


# ---- wide seam -------------------------------------------------------------------------------------------------------------
def _xyz(rng, n):
    x = np.zeros((n, 4), np.float32)
    x[:, :3] = rng.random((n, 3)) * 4
    if n:
        x[: n // 4, :3] = x[0, :3] + 0.02 * rng.standard_normal((n // 4, 3)).astype(np.float32)
    return x


def _wide_case(desc, n_scales, seed, n_sk=600, n_tk=700, rows=None, null_maps=False):
    rng = np.random.default_rng(seed)
    sx, tx = _xyz(rng, n_sk), _xyz(rng, n_tk)
    s_sc, t_sc, dim = [], [], synth.DESCRIPTORS[desc][0]
    for s in range(n_scales):
        ns, nt = rows[s] if rows else (n_sk - 50 * s, n_tk - 40 * s)
        smap = None if null_maps and ns == n_sk else np.sort(rng.choice(n_sk, ns, replace=False)).astype(np.int32)
        tmap = None if null_maps and nt == n_tk else np.sort(rng.choice(n_tk, nt, replace=False)).astype(np.int32)
        src, tgt, dim = synth.make_pair(desc, max(ns, 1), max(nt, 1), seed=1000 * seed + s, nan_frac=0.02)
        s_sc.append((np.ascontiguousarray(src[:ns]), smap))
        t_sc.append((np.ascontiguousarray(tgt[:nt]), tmap))
    pr = dict(src_scales=s_sc, tgt_scales=t_sc, src_kps_xyz=sx, tgt_kps_xyz=tx,
              iss_radius_src=np.float32(0.03 + 0.05 * rng.random()), iss_radius_tgt=np.float32(0.03 + 0.05 * rng.random()))
    return pr, rng.random(n_sk).astype(np.float32), rng.random(n_tk).astype(np.float32), dim


def _moved(pr, seed):
    rng = np.random.default_rng(seed)
    g = np.eye(4, dtype=np.float32)
    g[:3, 3] = 0.05 * rng.standard_normal(3)
    out = dict(pr)
    out["src_kps_moved"] = M.transform_keypoints(pr["src_kps_xyz"], g)
    out["tgt_kps_moved"] = M.transform_keypoints(pr["tgt_kps_xyz"], M.invert_guess(g))
    return out


def _to_dev(pr, dev):
    torch = _torch()
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    out = dict(pr)
    for side in ("src_scales", "tgt_scales"):
        out[side] = [(t(f), t(m)) for f, m in pr[side]]
    for key in ("src_kps_xyz", "tgt_kps_xyz", "src_kps_moved", "tgt_kps_moved"):
        if key in pr:
            out[key] = t(pr[key])
    return out


def _wide_cases(desc, n_scales, seed):
    cases = [_wide_case(desc, n_scales, seed + i) for i in range(3)]
    cases.append(_wide_case(desc, n_scales, seed + 10, n_sk=257, n_tk=256, rows=[(257, 256)] * n_scales, null_maps=True))
    cases.append(_wide_case(desc, 0, seed + 11))                                              # no scales
    cases.append(_wide_case(desc, n_scales, seed + 12, n_sk=0, rows=[(0, 600)] * n_scales))   # no source keypoints
    cases.append(_wide_case(desc, n_scales, seed + 13, n_sk=255, n_tk=1, rows=[(255, 1)] * n_scales))
    return cases


@gpu
@pytest.mark.parametrize("desc,k,n_scales", [("fpfh", 1, 1), ("fpfh", 2, 3), ("shot", 2, 2), ("rops", 5, 2)])
@pytest.mark.parametrize("mode", list(WMODES))
@pytest.mark.parametrize("radius", [None, 0.3, M.FLT_MAX])
def test_wide_batch_device_equals_host(desc, k, n_scales, mode, radius):
    torch = _torch()
    cases = _wide_cases(desc, n_scales, 20 + k)
    if radius is not None:
        cases = [(_moved(c[0], 7 + i), c[1], c[2], c[3]) for i, c in enumerate(cases)]
    pairs, ts, tt, dim = [c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], cases[0][3]
    b = _backend()
    dev_pairs = [_to_dev(pr, b.device) for pr in pairs]
    dts, dtt = [torch.from_numpy(a).to(b.device) for a in ts], [torch.from_numpy(a).to(b.device) for a in tt]
    with M.Context(0) as ctx:
        if radius is None:
            ref = ctx.match_wide_batch(k, WMODES[mode], pairs, dim, 40, DTHR, ts, tt)
            got = b.match_wide_batch(k, WMODES[mode], dev_pairs, dim, 40, DTHR, dts, dtt)
        else:
            ref = ctx.match_wide_local_batch(k, WMODES[mode], pairs, radius, dim, 40, DTHR, ts, tt)
            got = b.match_wide_local_batch(k, WMODES[mode], dev_pairs, radius, dim, 40, DTHR, dts, dtt)
    _same_records(got, ref)
    b.close()


# ---- launches, refusals, stream order -------------------------------------------------------------------------------------
@gpu
def test_launches_do_not_grow_with_pairs():
    src, tgt, dim = synth.make_pair("fpfh", 600, 650, seed=9, nan_frac=0.02)
    b = _backend()
    torch = _torch()
    ds, dt = torch.from_numpy(src).to(b.device), torch.from_numpy(tgt).to(b.device)
    thr = torch.rand(600, device=b.device)
    case = _moved(_wide_case("fpfh", 2, 30)[0], 3)
    dcase = _to_dev(case, b.device)
    counts = {}
    for n in (2, 32):
        calls = {
            "knn": lambda: b.knn_batch(2, [(ds, dt)] * n, dim),
            "match": lambda: b.match_batch(2, M.MODE_MUTUAL, [(ds, ds)] * n, dim, thr_src=[thr] * n, thr_tgt=[thr] * n),
            "wide": lambda: b.match_wide_batch(2, M.MODE_CLUSTER, [dcase] * n, dim),
            "local": lambda: b.match_wide_local_batch(2, M.MODE_MUTUAL, [dcase] * n, 0.3, dim),
        }
        for name, f in calls.items():
            b.ctx.reset_stats()
            f()
            counts.setdefault(name, []).append(b.ctx.stats()["launches"])
    for name, (a, c) in counts.items():
        assert a == c and a > 0, (name, a, c)
    b.close()


@gpu
def test_host_pointers_are_refused_by_name():
    torch = _torch()
    src, tgt, dim = synth.make_pair("fpfh", 300, 300, seed=11, nan_frac=0.0)
    host = np.ascontiguousarray(src)
    pinned = torch.from_numpy(src).pin_memory()
    with M.Context(0) as ref_ctx:
        ref_ctx.upload(0, src, dim)
        ref_ctx.upload(1, tgt, dim)
        ref = ref_ctx.match(1, M.MODE_MUTUAL)
    b = _backend()
    ctx = b.ctx
    ds, dt = torch.from_numpy(src).to(b.device), torch.from_numpy(tgt).to(b.device)
    out = torch.empty((1000, 4), dtype=torch.int32, device=b.device)
    idx = torch.empty((300, 1), dtype=torch.int32, device=b.device)
    dist = torch.empty((300, 1), dtype=torch.float32, device=b.device)
    cnt = torch.empty((300,), dtype=torch.int32, device=b.device)
    dthr = torch.rand(300, device=b.device)
    hthr = np.random.default_rng(1).random(300).astype(np.float32)
    S = 33 * 4
    for bad in (host.ctypes.data, pinned.data_ptr()):
        attempts = [
            (lambda: ctx.knn_batch_device(1, [(bad, 300, dt.data_ptr(), 300)], S, dim, idx.data_ptr(), dist.data_ptr(),
                                          cnt.data_ptr()), "pair 0: src"),
            (lambda: ctx.knn_batch_device(1, [(ds.data_ptr(), 300, dt.data_ptr(), 300)], S, dim, bad, dist.data_ptr(),
                                          cnt.data_ptr()), "idx"),
            (lambda: ctx.match_batch_device(1, M.MODE_MUTUAL, [(ds.data_ptr(), 300, bad, 300)], S, dim, out.data_ptr(), 1000),
             "pair 0: tgt"),
            (lambda: ctx.match_batch_device(1, M.MODE_MUTUAL, [(ds.data_ptr(), 300, dt.data_ptr(), 300)], S, dim, out.data_ptr(),
                                            1000, dthr.data_ptr(), hthr.ctypes.data), "thr_tgt"),
            (lambda: ctx.match_batch_device(1, M.MODE_MUTUAL, [(ds.data_ptr(), 300, dt.data_ptr(), 300)], S, dim, bad, 1000), "out"),
        ]
        wide = dict(scales=[(ds.data_ptr(), 300, 0, dt.data_ptr(), 300, 0)], n_src_kps=300, n_tgt_kps=300,
                    src_kps_xyz=ds.data_ptr(), tgt_kps_xyz=dt.data_ptr(), iss_radius_src=0.05, iss_radius_tgt=0.05)
        for field, where in (("src_kps_xyz", "pair 1: src_kps_xyz"), ("tgt_kps_xyz", "pair 1: tgt_kps_xyz")):
            attempts.append((lambda f=field: ctx.match_wide_batch_device(1, M.MODE_MUTUAL, [wide, dict(wide, **{f: bad})], S, dim, 16,
                                                                         out.data_ptr(), 1000), where))
        for i, where in ((0, "pair 1: scale 1: src_desc"), (2, "pair 1: scale 1: src_map"), (3, "pair 1: scale 1: tgt_desc"),
                         (5, "pair 1: scale 1: tgt_map")):
            sc = list(wide["scales"][0])
            sc[i] = bad
            attempts.append((lambda sc=sc: ctx.match_wide_batch_device(1, M.MODE_MUTUAL, [wide, dict(wide, scales=[wide["scales"][0], tuple(sc)])],
                                                                       S, dim, 16, out.data_ptr(), 1000), where))
        for field in ("src_kps_moved", "tgt_kps_moved"):
            loc = dict(wide, src_kps_moved=ds.data_ptr(), tgt_kps_moved=dt.data_ptr())
            attempts.append((lambda f=field, loc=loc: ctx.match_wide_local_batch_device(
                1, M.MODE_MUTUAL, [dict(loc, **{f: bad})], 0.3, S, dim, 16, out.data_ptr(), 1000), "pair 0: " + field))
        attempts.append((lambda: ctx.match_wide_batch_device(1, M.MODE_MUTUAL, [wide], S, dim, 16, out.data_ptr(), 1000, thr_src=bad,
                                                             thr_tgt=dthr.data_ptr()), "thr_src"))
        for f, where in attempts:
            ctx.reset_stats()
            with pytest.raises(M.B200MatchError, match="not device memory") as e:
                f()
            assert where in str(e.value) and "_device" in str(e.value), str(e.value)
            assert ctx.stats()["launches"] == 0
    # the context still answers a single pair correctly
    ctx.upload(0, src, dim)
    ctx.upload(1, tgt, dim)
    got = ctx.match(1, M.MODE_MUTUAL)
    assert got[0].tobytes() == ref[0].tobytes() and got[1] == ref[1]
    # GpuBackend refuses tensors that are not on its device before any library call
    with pytest.raises(M.B200MatchError, match="pair 0: src"):
        b.match_batch(1, M.MODE_MUTUAL, [(torch.from_numpy(src), dt)], dim)
    with pytest.raises(M.B200MatchError, match="same row stride"):
        b.knn_batch(1, [(ds, dt), (torch.from_numpy(synth.make_pair("shot", 10, 10)[0]).to(b.device)[:, :40], dt[:5])], dim)
    b.close()


@gpu
def test_bad_map_and_small_capacity_errors_match_host():
    torch = _torch()
    pr, ts, tt, dim = _wide_case("fpfh", 2, 40)
    bad = dict(pr)
    smap = pr["src_scales"][1][1].copy()
    smap[7] = 10 ** 6
    bad["src_scales"] = [pr["src_scales"][0], (pr["src_scales"][1][0], smap)]
    b = _backend()
    with M.Context(0) as ctx:
        with pytest.raises(M.B200MatchError) as eh:
            ctx.match_wide_batch(2, M.MODE_MUTUAL, [pr, bad], dim)
    with pytest.raises(M.B200MatchError) as ed:
        b.match_wide_batch(2, M.MODE_MUTUAL, [_to_dev(pr, b.device), _to_dev(bad, b.device)], dim)
    assert str(ed.value) == str(eh.value).replace("b200m_match_multiscale_batch", "b200m_match_multiscale_batch_device")
    # cap too small: the offsets are filled and the call fails, as the host form does
    with M.Context(0) as ctx:
        ref = ctx.match_wide_batch(2, M.MODE_MUTUAL, [pr, pr], dim)
    d = _to_dev(pr, b.device)
    out = torch.empty((4, 4), dtype=torch.int32, device=b.device)
    scales = [(f.data_ptr(), f.shape[0], 0 if m is None else m.data_ptr(), g.data_ptr(), g.shape[0], 0 if n is None else n.data_ptr())
              for (f, m), (g, n) in zip(d["src_scales"], d["tgt_scales"])]
    sc = (M._Scale * 2)(*[M._Scale(*[x or None for x in s]) for s in scales])
    arr = (M._WidePair * 2)()
    for i in range(2):
        arr[i] = M._WidePair(ctypes.cast(sc, ctypes.c_void_p), 2, d["src_kps_xyz"].data_ptr(), 600, d["tgt_kps_xyz"].data_ptr(), 700,
                             float(pr["iss_radius_src"]), float(pr["iss_radius_tgt"]))
    offs = np.zeros(3, np.uint64)
    p = M.Context._params(2, M.MODE_MUTUAL)
    b.use_torch_stream()
    rc = b.ctx._L.b200m_match_multiscale_batch_device(b.ctx._h, ctypes.byref(p), arr, 2, 33 * 4, dim, 16, 40, None, None,
                                                      out.data_ptr(), 4, offs.ctypes.data_as(ctypes.POINTER(ctypes.c_size_t)), None)
    assert rc != 0 and "output capacity too small" in b.ctx._L.b200m_last_error(b.ctx._h).decode()
    assert [int(x) for x in offs] == [0, len(ref[0][0]), len(ref[0][0]) + len(ref[1][0])]
    # the context still answers a single pair correctly afterwards
    src, tgt, dim1 = synth.make_pair("fpfh", 500, 400, seed=12)
    with M.Context(0) as c2:
        c2.upload(0, src, dim1)
        c2.upload(1, tgt, dim1)
        want = c2.match(1, M.MODE_MUTUAL)
    b.ctx.upload(0, src, dim1)
    b.ctx.upload(1, tgt, dim1)
    got = b.ctx.match(1, M.MODE_MUTUAL)
    assert got[0].tobytes() == want[0].tobytes() and got[1] == want[1]
    b.close()


@gpu
def test_inputs_written_by_torch_just_before_the_call():
    """no torch.cuda.synchronize between the op that writes the sets and the call: the library runs on torch's stream"""
    torch = _torch()
    b = _backend()
    src, tgt, dim = synth.make_pair("shot", 4000, 3000, seed=13, nan_frac=0.01)
    ds0, dt0 = torch.from_numpy(src).to(b.device), torch.from_numpy(tgt).to(b.device)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(b.device)
    with torch.cuda.stream(side):
        b.use_torch_stream()
        for _ in range(3):   # a long op right before, on the current (non-default) stream
            ds = (ds0 * 2.0) * 0.5
            dt = (dt0 * 2.0) * 0.5
        thr = torch.sigmoid(ds[:, 0]).contiguous()
        got = b.match_batch(2, M.MODE_MUTUAL, [(ds[:2000], dt), (ds[2000:], dt[:1000])], dim,
                            thr_src=[thr[:2000], thr[2000:]], thr_tgt=[thr[:3000], thr[1000:2000]])
        got = [(r.clone(), a) for r, a in got]
    torch.cuda.synchronize()
    h = thr.cpu().numpy()
    with M.Context(0) as ctx:
        ref = ctx.match_batch(2, M.MODE_MUTUAL, [(src[:2000], tgt), (src[2000:], tgt[:1000])], dim,
                              thr_src=[h[:2000], h[2000:]], thr_tgt=[h[:3000], h[1000:2000]])
    _same_records(got, ref)
    b.use_torch_stream()
    b.close()
