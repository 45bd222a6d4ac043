"""Device-resident and multi-GPU drivers of the matcher on torch tensors (HBM buffers, the current torch stream).

    GpuBackend      one b200m context working on torch device buffers (no host copies), single pairs and batches
    BatchPlan       a device batch call bound once (b200m_plan_*): run() only enqueues, so torch.cuda.graph can capture it
    ShardedMatcher  SURVEY 8e, one process per GPU: query-sharded / target-replicated matcher and the target-sharded kNN.
                    With a GpuBackend this is a THIN caller of the library -- partitioning, the NCCL exchange step and
                    the merge live in libb200match.so (csrc/multi.cu: b200m_match_sharded_device,
                    b200m_knn_target_sharded_device, b200m_upload_replicated); torch.distributed only carries the
                    128-byte communicator id to the ranks.  The same partitioning written out in Python over
                    torch.distributed collectives is kept for backends without native sharding: the CPU tests drive it
                    with gloo and a stand-in backend as an executable statement of the exchange protocol.
"""
import ctypes as C

import torch

from . import matcher as M


# below this many (query, train) pairs the row selection's host round trip costs more than the skipped rows save
MASKED_REVERSE_MIN_PAIRS = 10 ** 9


def shard_bounds(n, rank, world):
    """The library's row partition (b200m_shard_rows): rank r owns [r*R, min(n, (r+1)*R)), R = ceil(n / world) -- the
    all-gathered slots are then the row-major table of all rows."""
    per = (n + world - 1) // world
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


class GpuBackend:
    """kNN / filter / merge on device buffers through the C-ABI *_device entry points."""
    native_sharding = True    # partitioning + NCCL inside libb200match.so

    def __init__(self, device_index=0, precision=M.PREC_TC_F16, cand_cap=0):
        self.device = torch.device("cuda", device_index)
        torch.cuda.set_device(self.device)
        self.ctx = M.Context(device_index)
        self.precision = precision
        self.cand_cap = cand_cap
        self.use_torch_stream()

    def use_torch_stream(self):
        """Queue the library's work on torch's current stream.  torch reports the legacy default stream as
        handle 0, which the C-ABI reads as "use the context's own stream": pass cudaStreamLegacy (0x1) instead,
        otherwise torch's ops (NCCL waits, .item(), events) would not be ordered with the library's kernels."""
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream or 1)

    def close(self):
        self.ctx.close()

    @property
    def n(self):
        return self.ctx.n

    def attach_comm(self, rank, world, group=None):
        """Give the context its rank in an NCCL communicator of its own: rank 0 makes the id, torch.distributed carries
        the 128 bytes to the others (plumbing only)."""
        import torch.distributed as dist
        ident = torch.zeros(M.UNIQUE_ID_BYTES, dtype=torch.uint8)
        if rank == 0:
            ident = torch.frombuffer(bytearray(M.comm_unique_id()), dtype=torch.uint8).clone()
        on_dev = dist.get_backend(group) == "nccl"
        t = ident.to(self.device) if on_dev else ident
        dist.broadcast(t, src=0, group=group)
        self.ctx.comm_attach(world, rank, bytes(t.cpu().numpy().tobytes()))

    # -- descriptors ----------------------------------------------------------
    def upload_device(self, side, aos, dim, index_offset=0):
        """aos: float32 CUDA tensor [n, stride_floats] (AoS point structs resident in HBM)."""
        assert aos.is_cuda and aos.dtype == torch.float32 and aos.dim() == 2 and aos.stride(1) == 1
        self.ctx.upload_device(side, aos.data_ptr(), aos.shape[0], aos.stride(0) * 4, dim, index_offset)

    def upload_host(self, side, aos_host, dim, index_offset=0):
        """aos_host: float32 CPU tensor (pinned for a true async copy) [n, stride_floats]."""
        assert not aos_host.is_cuda and aos_host.dtype == torch.float32 and aos_host.stride(1) == 1
        self.ctx._ck(self.ctx._L.b200m_upload(self.ctx._h, side, aos_host.data_ptr(), aos_host.shape[0],
                                              aos_host.stride(0) * 4, dim, index_offset))
        self.ctx.n[side] = aos_host.shape[0]
        self.ctx.dim = dim
        return aos_host.shape[0] * aos_host.stride(0) * 4

    # -- kernels ----------------------------------------------------------------
    def knn(self, k, direction, row_begin, row_end):
        rows = row_end - row_begin
        idx = torch.empty((rows, k), dtype=torch.int32, device=self.device)
        dist = torch.empty((rows, k), dtype=torch.float32, device=self.device)
        cnt = torch.empty((rows,), dtype=torch.int32, device=self.device)
        if rows:
            self.ctx.knn_device(k, direction, row_begin, row_end, idx.data_ptr(), dist.data_ptr(), cnt.data_ptr(),
                                self.precision, self.cand_cap)
        return idx, dist, cnt

    def knn_masked(self, k, direction, row_begin, row_end, flags):
        """kNN of the rows of [row_begin, row_end) whose flag is set (uint8 CUDA tensor over ALL rows of the query side);
        the other rows get empty lists."""
        rows = row_end - row_begin
        idx = torch.empty((rows, k), dtype=torch.int32, device=self.device)
        dist = torch.empty((rows, k), dtype=torch.float32, device=self.device)
        cnt = torch.empty((rows,), dtype=torch.int32, device=self.device)
        if rows:
            self.ctx.knn_masked_device(k, direction, row_begin, row_end, flags.data_ptr(), idx.data_ptr(), dist.data_ptr(),
                                       cnt.data_ptr(), self.precision, self.cand_cap)
        return idx, dist, cnt

    def referenced_rows(self, k, fwd, n_flags, index_offset=0):
        """uint8 flags [n_flags]: 1 for every row of the other side that the k-lists `fwd` name."""
        flags = torch.zeros((n_flags,), dtype=torch.uint8, device=self.device)
        if fwd[0].shape[0]:
            self.ctx.mark_referenced_device(k, fwd[0].data_ptr(), fwd[2].data_ptr(), fwd[0].shape[0], index_offset,
                                            flags.data_ptr(), n_flags)
        return flags

    def filter(self, k, mode, row_begin, row_end, fwd, rev, n_rev_rows, ratio_thr=M.MATCHING_RATIO_THRESHOLD,
               distance_thr=M.FLT_MAX, thr_src=None, thr_tgt=None, want_avg=False):
        """-> (records int32 [cap, 4] (reinterpret as CORR_DTYPE), n_out uint64-as-int64 [1], avg float32 [1] or None)."""
        rows = row_end - row_begin
        kk = k if mode == M.MODE_MUTUAL else 1
        cap = max(rows * kk, 1)
        out = torch.empty((cap, 4), dtype=torch.int32, device=self.device)
        n_out = torch.zeros((1,), dtype=torch.int64, device=self.device)
        avg = torch.zeros((1,), dtype=torch.float32, device=self.device) if want_avg else None
        r = rev if rev is not None else (None, None, None)
        ptr = lambda t: 0 if t is None else t.data_ptr()
        self.ctx.filter_device(k, mode, row_begin, row_end, ptr(fwd[0]), ptr(fwd[1]), ptr(fwd[2]), ptr(r[0]), ptr(r[1]),
                               ptr(r[2]), n_rev_rows, out.data_ptr(), cap, n_out.data_ptr(), ptr(avg), ptr(thr_src),
                               ptr(thr_tgt), ratio_thr, distance_thr)
        return out, n_out, avg

    def merge(self, k, idx_in, dist_in, cnt_in):
        """idx_in/dist_in [n_lists, nq, k], cnt_in [n_lists, nq] -> the k best per query by (dist, idx)."""
        n_lists, nq = cnt_in.shape
        idx = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        dist = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        cnt = torch.empty((nq,), dtype=torch.int32, device=self.device)
        self.ctx.merge_device(k, n_lists, nq, idx_in.data_ptr(), dist_in.data_ptr(), cnt_in.data_ptr(), idx.data_ptr(),
                              dist.data_ptr(), cnt.data_ptr())
        return idx, dist, cnt

    def match_device(self, k, mode, ratio_thr=M.MATCHING_RATIO_THRESHOLD, distance_thr=M.FLT_MAX, want_avg=False):
        """Whole matcher call on one GPU, everything resident in HBM."""
        nq, nt = self.n
        fwd = self.knn(k, 0, 0, nq)
        rev = None
        if mode in (M.MODE_MUTUAL, M.MODE_RATIO_MUTUAL):
            if nq * nt >= MASKED_REVERSE_MIN_PAIRS:
                rev = self.knn_masked(k, 1, 0, nt, self.referenced_rows(k, fwd, nt))
            else:
                rev = self.knn(k, 1, 0, nt)
        return self.filter(k, mode, 0, nq, fwd, rev, nt if rev is not None else 0, ratio_thr, distance_thr,
                           want_avg=want_avg)

    # -- batches on device-resident sets (b200m_*_batch_device) ------------------------------------------
    def _check_rows(self, t, what, dtype=torch.float32, min_cols=1):
        """A 2-D tensor of `dtype` with unit column stride on this backend's device -> its row stride in elements (None
        for an empty set)."""
        if not isinstance(t, torch.Tensor) or t.dtype != dtype or t.dim() != 2 or t.device != self.device:
            raise M.B200MatchError("%s: must be a 2-D %s tensor on %s" % (what, dtype, self.device))
        if t.shape[1] < min_cols:
            raise M.B200MatchError("%s: rows must have at least %d columns" % (what, min_cols))
        if t.shape[0] == 0:
            return None
        if t.stride(1) != 1 and t.shape[1] > 1:
            raise M.B200MatchError("%s: the columns must be contiguous (unit column stride)" % what)
        return t.stride(0)

    def _check_vec(self, t, what, n, dtype):
        if not isinstance(t, torch.Tensor) or t.dtype != dtype or t.dim() != 1 or t.device != self.device:
            raise M.B200MatchError("%s: must be a 1-D %s tensor on %s" % (what, dtype, self.device))
        if t.shape[0] != n:
            raise M.B200MatchError("%s: %d entries, %d expected" % (what, t.shape[0], n))
        if n > 1 and t.stride(0) != 1:
            raise M.B200MatchError("%s: must be contiguous" % what)

    @staticmethod
    def _one_stride(strides, what):
        got = {st for st in strides if st is not None}
        if len(got) > 1:
            raise M.B200MatchError("%s: every set of the batch must have the same row stride (got %s)" % (what, sorted(got)))
        return got.pop() if got else None

    @staticmethod
    def _ptr(t):
        return t.data_ptr() if t is not None and t.numel() else 0

    def _set_pairs(self, pairs, dim):
        """[(src, tgt), ...] float32 CUDA tensors -> ([(ptr, n, ptr, n)], row stride in bytes)."""
        strides = []
        for i, pr in enumerate(pairs):
            if len(pr) != 2:
                raise M.B200MatchError("pair %d: a (source rows, target rows) tuple is needed" % i)
            for side, t in zip(("src", "tgt"), pr):
                strides.append(self._check_rows(t, "pair %d: %s" % (i, side), min_cols=dim))
        stride = self._one_stride(strides, "batch") or dim
        return [(self._ptr(s), s.shape[0], self._ptr(t), t.shape[0]) for s, t in pairs], stride * 4

    def _thresholds(self, thr_src, thr_tgt, counts):
        """one 1-D float32 tensor per pair and side -> the two concatenations (device tensors) or (None, None)."""
        if (thr_src is None) != (thr_tgt is None):
            raise M.B200MatchError("give both threshold lists or neither")
        if thr_src is None:
            return None, None
        if len(thr_src) != len(counts) or len(thr_tgt) != len(counts):
            raise M.B200MatchError("one threshold array per pair and side")
        for i, (ns, nt) in enumerate(counts):
            self._check_vec(thr_src[i], "pair %d: thr_src" % i, ns, torch.float32)
            self._check_vec(thr_tgt[i], "pair %d: thr_tgt" % i, nt, torch.float32)
        pad = [torch.zeros(1, dtype=torch.float32, device=self.device)]
        return torch.cat(list(thr_src) + pad), torch.cat(list(thr_tgt) + pad)

    def knn_batch(self, k, pairs, dim):
        """b200m_knn_batch_device on [(source rows, target rows), ...] (float32 CUDA tensors [n, >= dim], unit column
        stride, one row stride in the batch; row slices of a larger tensor and one tensor in many pairs are fine).
        -> one (idx, dist, cnt) CUDA tensor view per pair, equal to Context.knn_batch on the same data."""
        ptrs, stride = self._set_pairs(pairs, dim)
        total = sum(p[1] for p in ptrs)
        idx = torch.empty((total, k), dtype=torch.int32, device=self.device)
        dist = torch.empty((total, k), dtype=torch.float32, device=self.device)
        cnt = torch.empty((total,), dtype=torch.int32, device=self.device)
        self.use_torch_stream()
        self.ctx.knn_batch_device(k, ptrs, stride, dim, self._ptr(idx), self._ptr(dist), self._ptr(cnt), self.precision,
                                  self.cand_cap)
        out, a = [], 0
        for p in ptrs:
            out.append((idx[a:a + p[1]], dist[a:a + p[1]], cnt[a:a + p[1]]))
            a += p[1]
        return out

    def match_batch(self, k, mode, pairs, dim, ratio_thr=M.MATCHING_RATIO_THRESHOLD, distance_thr=M.FLT_MAX, thr_src=None,
                    thr_tgt=None):
        """b200m_match_batch_device: -> one (records int32 [n, 4] CUDA view (CORR_DTYPE layout), average) per pair, equal
        to Context.match_batch on the same data.  thr_src / thr_tgt: None or one 1-D float32 CUDA tensor per pair."""
        ptrs, stride = self._set_pairs(pairs, dim)
        ts, tt = self._thresholds(thr_src, thr_tgt, [(p[1], p[3]) for p in ptrs])
        kk = k if mode == M.MODE_MUTUAL else 1
        cap = max(sum(p[1] for p in ptrs) * kk, 1)
        out = torch.empty((cap, 4), dtype=torch.int32, device=self.device)
        self.use_torch_stream()
        offsets, avg = self.ctx.match_batch_device(k, mode, ptrs, stride, dim, out.data_ptr(), cap, self._ptr(ts), self._ptr(tt),
                                                   ratio_thr, distance_thr, self.precision, self.cand_cap)
        return [(out[int(offsets[i]):int(offsets[i + 1])], float(avg[i])) for i in range(len(pairs))]

    # -- batch plans (b200m_plan_*): bound once, then enqueued without the host ----------------------------------------
    def plan_knn_batch(self, k, pairs, dim):
        """A BatchPlan of knn_batch over `pairs` (as knn_batch takes them).  The plan binds the tensors themselves: run()
        answers on whatever they hold when it runs.  Outputs: plan.idx [sum n_src, k], plan.dist, plan.cnt [sum n_src]."""
        ptrs, stride = self._set_pairs(pairs, dim)
        total = sum(p[1] for p in ptrs)
        out = dict(idx=torch.empty((total, k), dtype=torch.int32, device=self.device),
                   dist=torch.empty((total, k), dtype=torch.float32, device=self.device),
                   cnt=torch.empty((total,), dtype=torch.int32, device=self.device))
        p = M.Context._params(k, M.MODE_KNN_ONLY, precision=self.precision, cand_cap=self.cand_cap)
        arr = M.Context._device_pairs(ptrs)
        make = lambda h: self.ctx._L.b200m_plan_knn_batch(self.ctx._h, C.byref(p), arr, len(ptrs), stride, dim,
                                                          self._ptr(out["idx"]), self._ptr(out["dist"]),
                                                          self._ptr(out["cnt"]), h)
        return BatchPlan(self, ptrs, list(pairs), out, make)

    def plan_match_batch(self, k, mode, pairs, dim, cap=None, thr_src=None, thr_tgt=None, ratio_thr=M.MATCHING_RATIO_THRESHOLD,
                         distance_thr=M.FLT_MAX):
        """A BatchPlan of match_batch over `pairs`.  thr_src / thr_tgt: None or one 1-D float32 tensor per pair, bound in
        place, so they must be consecutive slices of one tensor per side in pair order (torch.split of it).  cap: records
        the plan writes (default sum n_src * (k if MUTUAL else 1), enough for any data).  Outputs: plan.records int32
        [cap, 4] (CORR_DTYPE layout), plan.offsets int64 [n_pairs + 1], plan.avg float32 [n_pairs], plan.n_out int64 [1]
        (records found; above cap the records were truncated)."""
        ptrs, stride = self._set_pairs(pairs, dim)
        if (thr_src is None) != (thr_tgt is None):
            raise M.B200MatchError("give both threshold lists or neither")
        keep = list(pairs)
        thr = [0, 0]
        if thr_src is not None:
            for side, (thrs, col) in enumerate(((thr_src, 1), (thr_tgt, 3))):
                if len(thrs) != len(ptrs):
                    raise M.B200MatchError("one threshold array per pair and side")
                thr[side], t = self._bound_thresholds(thrs, [q[col] for q in ptrs], "thr_src" if side == 0 else "thr_tgt")
                keep.append(t)
        kk = k if mode == M.MODE_MUTUAL else 1
        cap = max(sum(q[1] for q in ptrs) * kk, 1) if cap is None else int(cap)
        out = dict(records=torch.empty((cap, 4), dtype=torch.int32, device=self.device),
                   offsets=torch.zeros((len(ptrs) + 1,), dtype=torch.int64, device=self.device),
                   avg=torch.empty((len(ptrs),), dtype=torch.float32, device=self.device),
                   n_out=torch.zeros((1,), dtype=torch.int64, device=self.device))
        p = M.Context._params(k, mode, ratio_thr, distance_thr, self.precision, self.cand_cap)
        arr = M.Context._device_pairs(ptrs)
        make = lambda h: self.ctx._L.b200m_plan_match_batch(self.ctx._h, C.byref(p), arr, len(ptrs), stride, dim, thr[0], thr[1],
                                                            self._ptr(out["records"]), cap, self._ptr(out["offsets"]),
                                                            self._ptr(out["avg"]), self._ptr(out["n_out"]), h)
        return BatchPlan(self, ptrs, keep, out, make)

    def _bound_thresholds(self, thrs, counts, what):
        """per-pair threshold tensors that lie back to back in one tensor -> (device pointer of the first, what to keep)"""
        base, expect = None, None
        for i, (t, n) in enumerate(zip(thrs, counts)):
            self._check_vec(t, "pair %d: %s" % (i, what), n, torch.float32)
            if n == 0:
                continue
            if base is None:
                base = expect = t.data_ptr()
            if t.data_ptr() != expect:
                raise M.B200MatchError("%s: a plan binds the thresholds in place; they must be consecutive slices of one tensor "
                                       "in pair order (pair %d is not)" % (what, i))
            expect += 4 * n
        if base is None:   # no rows on this side: any device word stands for the empty array
            t = torch.zeros((1,), dtype=torch.float32, device=self.device)
            return t.data_ptr(), t
        return base, list(thrs)

    def match_wide_batch(self, k, mode, pairs, dim=None, cluster_k=M.MATCHING_CLUSTER_K, distance_thr=M.FLT_MAX, thr_src=None,
                         thr_tgt=None):
        """b200m_match_multiscale_batch_device: the dicts of Context.match_wide_batch (src_scales / tgt_scales = lists of
        (features, index map or None), src_kps_xyz, tgt_kps_xyz, iss_radius_src, iss_radius_tgt) with CUDA tensors:
        float32 features and coordinates [n, >= 3], int32 maps.  -> one (records view, average) per pair."""
        return self._wide_batch(k, mode, pairs, None, dim, cluster_k, distance_thr, thr_src, thr_tgt)

    def match_wide_local_batch(self, k, mode, pairs, match_search_radius, dim=None, cluster_k=M.MATCHING_CLUSTER_K,
                               distance_thr=M.FLT_MAX, thr_src=None, thr_tgt=None):
        """b200m_match_multiscale_local_batch_device: match_wide_batch's dicts plus src_kps_moved / tgt_kps_moved (the
        latter may be None in ONE_SIDED mode), as Context.match_wide_local_batch takes them."""
        return self._wide_batch(k, mode, pairs, float(match_search_radius), dim, cluster_k, distance_thr, thr_src, thr_tgt)

    def _wide_args(self, pairs, radius, dim):
        """match_wide_batch's dicts -> (match_wide_batch_device's dicts, [(n_src_kps, n_tgt_kps)], descriptor row stride in
        bytes, dim, keypoint row stride in bytes)"""
        fs = [dict(pr) if isinstance(pr, dict) else dict(zip(M.Context._WIDE_FIELDS, pr)) for pr in pairs]
        desc_strides, xyz_strides, width, out_pairs, counts = [], [], None, [], []
        for i, f in enumerate(fs):
            if len(f["src_scales"]) != len(f["tgt_scales"]):
                raise M.B200MatchError("pair %d: need the same number of scales on both sides" % i)
            scales = []
            for s, ((sf, sm), (tf, tm)) in enumerate(zip(f["src_scales"], f["tgt_scales"])):
                for side, t, m in (("src", sf, sm), ("tgt", tf, tm)):
                    desc_strides.append(self._check_rows(t, "pair %d: scale %d: %s features" % (i, s, side)))
                    if width is not None and t.shape[1] != width:
                        raise M.B200MatchError("pair %d: scale %d: every descriptor row must have the same length" % (i, s))
                    width = t.shape[1]
                    if m is not None:
                        self._check_vec(m, "pair %d: scale %d: %s map" % (i, s, side), t.shape[0], torch.int32)
                scales.append((self._ptr(sf), sf.shape[0], self._ptr(sm), self._ptr(tf), tf.shape[0], self._ptr(tm)))
            xs = {}
            for key in ("src_kps_xyz", "tgt_kps_xyz") + (("src_kps_moved", "tgt_kps_moved") if radius is not None else ()):
                x = f.get(key)
                if x is not None:
                    xyz_strides.append(self._check_rows(x, "pair %d: %s" % (i, key), min_cols=3))
                xs[key] = x
            if xs["tgt_kps_xyz"] is None:
                raise M.B200MatchError("pair %d: tgt_kps_xyz is needed" % i)
            ns = xs["src_kps_xyz"].shape[0] if xs["src_kps_xyz"] is not None else int(f.get("n_src_kps", 0))
            nt = xs["tgt_kps_xyz"].shape[0]
            if radius is not None:
                for key, n in (("src_kps_moved", ns), ("tgt_kps_moved", nt)):
                    if xs[key] is not None and xs[key].shape[0] != n:
                        raise M.B200MatchError("pair %d: moved keypoints must have the rows of the unmoved ones" % i)
            counts.append((ns, nt))
            d = dict(scales=scales, n_src_kps=ns, n_tgt_kps=nt, iss_radius_src=float(f["iss_radius_src"]),
                     iss_radius_tgt=float(f["iss_radius_tgt"]))
            for key, x in xs.items():
                d[key] = self._ptr(x)
            out_pairs.append(d)
        width = width or int(dim or 1)
        dim = int(dim or width)
        if dim > width:
            raise M.B200MatchError("dim exceeds the row length")
        stride = self._one_stride(desc_strides, "descriptor sets") or width
        xyz_stride = self._one_stride(xyz_strides, "keypoint coordinates") or 4
        return out_pairs, counts, stride * 4, dim, xyz_stride * 4

    def _wide_batch(self, k, mode, pairs, radius, dim, cluster_k, distance_thr, thr_src, thr_tgt):
        out_pairs, counts, stride, dim, xyz_stride = self._wide_args(pairs, radius, dim)
        ts, tt = self._thresholds(thr_src, thr_tgt, counts)
        cap = max(sum(ns for ns, _ in counts), 1)
        out = torch.empty((cap, 4), dtype=torch.int32, device=self.device)
        self.use_torch_stream()
        if radius is None:
            offsets, avg = self.ctx.match_wide_batch_device(k, mode, out_pairs, stride, dim, xyz_stride, out.data_ptr(), cap,
                                                            cluster_k, distance_thr, self._ptr(ts), self._ptr(tt), self.precision,
                                                            self.cand_cap)
        else:
            offsets, avg = self.ctx.match_wide_local_batch_device(k, mode, out_pairs, radius, stride, dim, xyz_stride,
                                                                  out.data_ptr(), cap, cluster_k, distance_thr, self._ptr(ts),
                                                                  self._ptr(tt))
        return [(out[int(offsets[i]):int(offsets[i + 1])], float(avg[i])) for i in range(len(pairs))]

    def plan_match_wide_batch(self, k, mode, pairs, dim=None, cluster_k=M.MATCHING_CLUSTER_K, distance_thr=M.FLT_MAX,
                              thr_src=None, thr_tgt=None, cap=None):
        """A BatchPlan of match_wide_batch over `pairs` (the same dicts).  Every tensor in them is bound in place; thr_src /
        thr_tgt: None or one 1-D float32 tensor per pair of its keypoints, consecutive slices of one tensor per side.  cap:
        records the plan writes (default the total source keypoints, enough for any data).  Outputs as plan_match_batch's,
        plus plan.status int64 [1]: the bad-map key (-1, i.e. ~0, when clean; results() raises on any other)."""
        return self._plan_wide(k, mode, pairs, None, dim, cluster_k, distance_thr, thr_src, thr_tgt, cap)

    def plan_match_wide_local_batch(self, k, mode, pairs, match_search_radius, dim=None, cluster_k=M.MATCHING_CLUSTER_K,
                                    distance_thr=M.FLT_MAX, thr_src=None, thr_tgt=None, cap=None):
        """A BatchPlan of match_wide_local_batch over `pairs` (its dicts, moved keypoints included)."""
        return self._plan_wide(k, mode, pairs, float(match_search_radius), dim, cluster_k, distance_thr, thr_src, thr_tgt, cap)

    def _plan_wide(self, k, mode, pairs, radius, dim, cluster_k, distance_thr, thr_src, thr_tgt, cap):
        out_pairs, counts, stride, dim, xyz_stride = self._wide_args(pairs, radius, dim)
        if (thr_src is None) != (thr_tgt is None):
            raise M.B200MatchError("give both threshold lists or neither")
        keep = list(pairs)
        thr = [0, 0]
        if thr_src is not None:
            for side, thrs in enumerate((thr_src, thr_tgt)):
                if len(thrs) != len(counts):
                    raise M.B200MatchError("one threshold array per pair and side")
                thr[side], t = self._bound_thresholds(thrs, [c[side] for c in counts], "thr_src" if side == 0 else "thr_tgt")
                keep.append(t)
        cap = max(sum(ns for ns, _ in counts), 1) if cap is None else int(cap)
        n = len(counts)
        out = dict(records=torch.empty((cap, 4), dtype=torch.int32, device=self.device),
                   offsets=torch.zeros((n + 1,), dtype=torch.int64, device=self.device),
                   avg=torch.empty((n,), dtype=torch.float32, device=self.device),
                   n_out=torch.zeros((1,), dtype=torch.int64, device=self.device),
                   status=torch.full((1,), -1, dtype=torch.int64, device=self.device))
        p = M.Context._params(k, mode, distance_thr=distance_thr, precision=self.precision, cand_cap=self.cand_cap)
        arr, locs, _scales = M.Context._wide_device_pairs(out_pairs, radius is not None)
        L, ptr = self.ctx._L, self._ptr
        tail = (thr[0], thr[1], ptr(out["records"]), cap, ptr(out["offsets"]), ptr(out["avg"]), ptr(out["n_out"]), ptr(out["status"]))
        if radius is None:
            make = lambda h: L.b200m_plan_match_multiscale_batch(self.ctx._h, C.byref(p), arr, n, stride, dim, xyz_stride,
                                                                 int(cluster_k), *tail, h)
        else:
            make = lambda h: L.b200m_plan_match_multiscale_local_batch(self.ctx._h, C.byref(p), arr, locs, n, stride, dim,
                                                                       xyz_stride, int(cluster_k), radius, *tail, h)
        return BatchPlan(self, [(0, ns, 0, nt) for ns, nt in counts], keep, out, make)


class BatchPlan:
    """A device batch call bound once (GpuBackend.plan_knn_batch / plan_match_batch / plan_match_wide_batch /
    plan_match_wide_local_batch).  run() enqueues it on torch's current stream with no host round trip, allocation or copy,
    so it may be captured in torch.cuda.graph; a run or a replay answers on what the bound input tensors hold at that time.
    The outputs are the plan's static tensors (attributes)."""

    def __init__(self, backend, ptrs, keep, outputs, make):
        self._L = backend.ctx._L
        self._h = None
        self.status = None           # matcher-class plans: the bad-map key
        self.device = backend.device
        self.counts = [(q[1], q[3]) for q in ptrs]
        self._keep = keep            # the bound tensors stay alive as long as the plan
        self.kind = "match" if "records" in outputs else "knn"
        for name, t in outputs.items():
            setattr(self, name, t)
        backend.use_torch_stream()   # creation runs the batch once on the context's stream: after torch's writes
        h = C.c_void_p()
        if make(C.byref(h)) != 0:
            raise M.B200MatchError(self._L.b200m_last_error(backend.ctx._h).decode())
        self._h = h

    def run(self):
        """Enqueue the batch on torch's current stream (nothing is returned; the outputs are the plan's tensors)."""
        if self._L.b200m_plan_run(self._h, torch.cuda.current_stream(self.device).cuda_stream) != 0:
            raise M.B200MatchError(self._L.b200m_plan_last_error(self._h).decode())

    def results(self):
        """Synchronise torch's current stream and split the outputs into per-pair views: knn -> [(idx, dist, cnt)], match
        -> [(records int32 [n, 4], average)], as GpuBackend.knn_batch / match_batch return them."""
        torch.cuda.current_stream(self.device).synchronize()
        out, a = [], 0
        if self.kind == "knn":
            for ns, _ in self.counts:
                out.append((self.idx[a:a + ns], self.dist[a:a + ns], self.cnt[a:a + ns]))
                a += ns
            return out
        if self.status is not None:
            msg = self._L.b200m_plan_status_error(self._h, int(self.status.item()) & 0xFFFFFFFFFFFFFFFF)
            if msg is not None:
                raise M.B200MatchError(msg.decode())
        n = int(self.n_out.item())
        if n > self.records.shape[0]:
            raise M.B200MatchError("plan output capacity too small (%d correspondences)" % n)
        offsets = self.offsets.cpu().tolist()
        avg = self.avg.cpu().tolist()
        return [(self.records[offsets[i]:offsets[i + 1]], avg[i]) for i in range(len(self.counts))]

    def close(self):
        if self._h:
            self._L.b200m_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def records_to_numpy(records, n_out):
    """int32 [cap,4] device tensor + count -> CORR_DTYPE host array."""
    n = int(n_out.item())
    return records[:n].contiguous().cpu().numpy().view(M.CORR_DTYPE).reshape(-1)


class ShardedMatcher:
    """One process per GPU.  `dist` is torch.distributed (or None for a single process)."""

    def __init__(self, backend, rank=0, world=1, group=None):
        self.b = backend
        self.rank, self.world, self.group = rank, world, group
        self.native = world > 1 and getattr(backend, "native_sharding", False)
        if self.native:
            backend.attach_comm(rank, world, group)

    # -- collectives ------------------------------------------------------------
    def _all_gather_rows(self, t, n_total):
        """All-gather row-sharded tensors (shard_bounds layout) into the full [n_total, ...] tensor."""
        if self.world == 1:
            return t
        import torch.distributed as dist
        max_rows = (n_total + self.world - 1) // self.world
        pad = torch.zeros((max_rows,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        pad[:t.shape[0]] = t
        out = torch.empty((self.world * max_rows,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, pad, group=self.group)
        if n_total % self.world == 0:
            return out
        parts = []
        for r in range(self.world):
            lo, hi = shard_bounds(n_total, r, self.world)
            parts.append(out[r * max_rows:r * max_rows + (hi - lo)])
        return torch.cat(parts, 0)

    # -- descriptor replication over NVLink instead of PCIe ---------------------------
    def upload_host_sharded(self, side, aos_host, dim, index_offset=0):
        """Replicate a HOST descriptor set on every rank: rank r copies only its 1/world slice over PCIe and the
        slices are all-gathered over NVLink (8 ranks pulling the whole set through the host's memory system at
        once is what limits the end-to-end rate of a replicated run).  aos_host: pinned float32 [n, stride_floats]."""
        if self.world == 1:
            return self.b.upload_host(side, aos_host, dim, index_offset)
        n = aos_host.shape[0]
        if self.native:
            assert index_offset == 0
            c = self.b.ctx
            c._ck(c._L.b200m_upload_replicated(c._h, side, aos_host.data_ptr(), n, aos_host.stride(0) * 4, dim))
            c.n[side], c.dim = n, dim
            lo, hi = shard_bounds(n, self.rank, self.world)
            return (hi - lo) * aos_host.stride(0) * 4
        lo, hi = shard_bounds(n, self.rank, self.world)
        shard = aos_host[lo:hi].to(self.b.device, non_blocking=True)
        full = self._all_gather_rows(shard, n)
        self.b.upload_device(side, full, dim, index_offset)     # the pack kernel reads `full` on this same stream
        return (hi - lo) * aos_host.stride(0) * 4               # bytes this rank moved host -> device

    # -- query-sharded, target replicated (SURVEY 8e, configs C3/C4) -----------------
    def match_query_sharded(self, k, mode, ratio_thr=M.MATCHING_RATIO_THRESHOLD, distance_thr=M.FLT_MAX):
        """Both descriptor sets are resident on every rank.  Returns this rank's slice of the
        correspondence list (records, n_out): concatenating the slices in rank order gives the
        single-GPU output (ascending index_query)."""
        nq, nt = self.b.n
        q0, q1 = shard_bounds(nq, self.rank, self.world)
        if self.native:
            cap = max((q1 - q0) * (k if mode == M.MODE_MUTUAL else 1), 1)
            out = torch.empty((cap, 4), dtype=torch.int32, device=self.b.device)
            n_out = torch.zeros((1,), dtype=torch.int64, device=self.b.device)
            self.b.ctx.match_sharded_device(k, mode, out.data_ptr(), cap, n_out.data_ptr(), ratio_thr=ratio_thr,
                                            distance_thr=distance_thr, precision=self.b.precision, cand_cap=self.b.cand_cap)
            return out, n_out, None
        fwd = self.b.knn(k, 0, q0, q1)
        rev = None
        if mode in (M.MODE_MUTUAL, M.MODE_RATIO_MUTUAL):
            t0, t1 = shard_bounds(nt, self.rank, self.world)
            if nq * nt >= MASKED_REVERSE_MIN_PAIRS:
                # the mutual test reads rev[j] only for targets j that a forward list names: every rank marks the ones its
                # own source rows name, the flags are max-reduced (nt bytes), and the reverse pass skips the rest
                flags = self.b.referenced_rows(k, fwd, nt)
                if self.world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(flags, op=dist.ReduceOp.MAX, group=self.group)
                r = self.b.knn_masked(k, 1, t0, t1, flags)
            else:
                r = self.b.knn(k, 1, t0, t1)
            rev = tuple(self._all_gather_rows(x, nt) for x in r)     # the path's one exchange step
        return self.b.filter(k, mode, q0, q1, fwd, rev, nt if rev is not None else 0, ratio_thr, distance_thr)

    def gather_records(self, records, n_out):
        """Concatenate every rank's correspondence slice in rank order on all ranks -> (records, n)."""
        if self.world == 1:
            return records[:int(n_out.item())], int(n_out.item())
        import torch.distributed as dist
        counts = torch.empty((self.world,), dtype=torch.int64, device=records.device)
        dist.all_gather_into_tensor(counts, n_out.to(torch.int64), group=self.group)
        counts_h = counts.cpu().tolist()
        mx = max(max(counts_h), 1)
        pad = torch.zeros((mx, 4), dtype=records.dtype, device=records.device)
        pad[:counts_h[self.rank]] = records[:counts_h[self.rank]]
        out = torch.empty((self.world * mx, 4), dtype=records.dtype, device=records.device)
        dist.all_gather_into_tensor(out, pad, group=self.group)
        parts = [out[r * mx:r * mx + counts_h[r]] for r in range(self.world)]
        return torch.cat(parts, 0), sum(counts_h)

    # -- target-sharded (config C5): each rank holds a slice of the target set ---------
    def knn_target_sharded(self, k):
        """The backend's side 1 holds THIS rank's target shard (uploaded with index_offset = shard start), side 0
        all queries.  Exact local top-k with global indices -> all-gather -> merge kernel (canonical tie rule)."""
        nq = self.b.n[0]
        if self.native:
            idx = torch.empty((nq, k), dtype=torch.int32, device=self.b.device)
            dist_ = torch.empty((nq, k), dtype=torch.float32, device=self.b.device)
            cnt = torch.empty((nq,), dtype=torch.int32, device=self.b.device)
            self.b.ctx.knn_target_sharded_device(k, idx.data_ptr(), dist_.data_ptr(), cnt.data_ptr(), self.b.precision,
                                                 self.b.cand_cap)
            return idx, dist_, cnt
        local = self.b.knn(k, 0, 0, nq)
        if self.world == 1:
            return local
        import torch.distributed as dist
        gathered = []
        for x in local:
            out = torch.empty((self.world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
            dist.all_gather_into_tensor(out, x.contiguous(), group=self.group)
            gathered.append(out.view((self.world,) + tuple(x.shape)))
        return self.b.merge(k, gathered[0], gathered[1], gathered[2])
