"""Host-side mirror of the reference's matcher interface on top of libb200match.so (C-ABI,
include/b200match.h).  Names and argument meaning follow the reference:

    match_bf(query, train, parameters)            <- matchBF<FeatureT>            include/matching.h:594-634
    match_flann / match_local(radius=inf)         <- matchFLANN / matchLocal      :562-592 / :637-678 (same result set)
    OneSidedMatcher / LeftToRightMatcher / RatioMatcher(.match(), .get_average_distance(), .get_class_name())
                                                  <- include/matching.h:385-478, :25-42
    get_feature_based_matcher_from_parameters     <- src/matching.cpp:21-76
    AlignmentParameters (hot-path subset)         <- include/common.h:135-163

Descriptors are float32 arrays [n, stride_floats] whose leading `dim` columns are the
descriptor -- the AoS layout PCL hands to the reference (`&cloud.points[0]`, `sizeof(FeatureT)`):
FPFH-33 (33 floats), RoPS-135 (135), SHOT-352 (361: descriptor + rf[9]), USC-1960 (1969: descriptor + rf[9]); any
dim up to 2048.  There is no CPU path here: without the CUDA library and a B200 every call raises.
"""
import atexit
import contextlib
import ctypes as C
import dataclasses
import os
import threading
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libb200match.so")

CORR_DTYPE = np.dtype([("index_query", "<i4"), ("index_match", "<i4"),
                       ("distance", "<f4"), ("threshold", "<f4")])

MODE_KNN_ONLY, MODE_ONE_SIDED, MODE_MUTUAL, MODE_RATIO, MODE_RATIO_MUTUAL, MODE_CLUSTER = 0, 1, 2, 3, 4, 5
PREC_TC_F16, PREC_F32_EXACT = 0, 2
SHARD_QUERY, SHARD_TARGET = 0, 1
UNIQUE_ID_BYTES = 128

# reference constants (include/common.h:50-51, :42, :45)
MATCHING_RATIO_THRESHOLD = 1.1
MATCHING_RATIO_K = 2
MATCHING_CLUSTER_K, MATCHING_CLUSTER_THRESHOLD = 40, 0.95   # include/common.h:52-53
MATCHING_ONE_SIDED, MATCHING_LEFT_TO_RIGHT, MATCHING_RATIO, MATCHING_CLUSTER = "one_sided", "lr", "ratio", "cluster"
FLT_MAX = float(np.finfo(np.float32).max)


class B200MatchError(RuntimeError):
    """== the std::runtime_error thrown by the reference's rassert (include/utils.h:9)."""


class _Params(C.Structure):
    _fields_ = [("k", C.c_int32), ("mode", C.c_int32), ("ratio_thr", C.c_float), ("distance_thr", C.c_float),
                ("precision", C.c_int32), ("cand_cap", C.c_int32), ("n_gpus", C.c_int32), ("shard", C.c_int32)]


class _Scale(C.Structure):
    _fields_ = [("src_desc", C.c_void_p), ("n_src", C.c_size_t), ("src_map", C.c_void_p),
                ("tgt_desc", C.c_void_p), ("n_tgt", C.c_size_t), ("tgt_map", C.c_void_p)]


class _Pair(C.Structure):
    """b200m_pair: one (source, target) pair of a batch call (host pointers)."""
    _fields_ = [("src", C.c_void_p), ("n_src", C.c_size_t), ("tgt", C.c_void_p), ("n_tgt", C.c_size_t)]


class _WidePair(C.Structure):
    """b200m_wide_pair: one (source, target) cloud pair of b200m_match_multiscale_batch (host pointers)."""
    _fields_ = [("scales", C.c_void_p), ("n_scales", C.c_int), ("src_kps_xyz", C.c_void_p), ("n_src_kps", C.c_size_t),
                ("tgt_kps_xyz", C.c_void_p), ("n_tgt_kps", C.c_size_t), ("iss_radius_src", C.c_float),
                ("iss_radius_tgt", C.c_float)]


class _LocalPair(C.Structure):
    """b200m_local_pair: the moved keypoints of one pair of b200m_match_multiscale_local_batch (host pointers)."""
    _fields_ = [("src_kps_moved", C.c_void_p), ("tgt_kps_moved", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("ms_pack", C.c_double), ("ms_prepare", C.c_double), ("ms_candidates", C.c_double),
                ("ms_rerank", C.c_double), ("ms_fallback", C.c_double), ("ms_filter", C.c_double),
                ("launches", C.c_int64), ("candidate_launches", C.c_int64), ("rows_total", C.c_int64),
                ("rows_flagged", C.c_int64), ("candidates", C.c_int64), ("rows_answered", C.c_int64),
                ("pairs_scored", C.c_int64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


EXPORTS = ["b200m_create", "b200m_destroy", "b200m_last_error", "b200m_set_stream", "b200m_sync",
           "b200m_set_profiling", "b200m_get_stats", "b200m_reset_stats", "b200m_upload", "b200m_upload_device",
           "b200m_knn", "b200m_knn_device", "b200m_match", "b200m_filter_device", "b200m_merge_device",
           "b200m_version", "b200m_debug_operands", "b200m_debug_tc_tile", "b200m_debug_candidate_lists", "b200m_multiscale_begin",
           "b200m_multiscale_add", "b200m_multiscale_vote", "b200m_multiscale_add_device", "b200m_multiscale_vote_device", "b200m_match_cluster",
           "b200m_cluster_filter_device", "b200m_knn3d_device", "b200m_knn_local", "b200m_knn_local_device", "b200m_mark_referenced_device", "b200m_knn_masked_device",
           "b200m_match_multiscale", "b200m_comm_unique_id", "b200m_comm_attach", "b200m_comm_rank", "b200m_shard_rows",
           "b200m_upload_replicated", "b200m_match_sharded", "b200m_match_sharded_device", "b200m_knn_target_sharded_device",
           "b200m_create_multi", "b200m_destroy_multi", "b200m_group_last_error", "b200m_group_size", "b200m_group_ctx",
           "b200m_group_upload", "b200m_group_upload_sharded", "b200m_group_match", "b200m_group_knn", "b200m_knn_batch",
           "b200m_match_batch", "b200m_match_multiscale_batch", "b200m_match_multiscale_local_batch", "b200m_knn_batch_device",
           "b200m_match_batch_device", "b200m_match_multiscale_batch_device", "b200m_match_multiscale_local_batch_device",
           "b200m_plan_knn_batch", "b200m_plan_match_batch", "b200m_plan_run", "b200m_plan_destroy", "b200m_plan_last_error",
           "b200m_plan_match_multiscale_batch", "b200m_plan_match_multiscale_local_batch", "b200m_plan_status_error",
           "b200m_plan_knn_batch_rows", "b200m_plan_match_batch_rows", "b200m_plan_match_multiscale_batch_rows",
           "b200m_plan_match_multiscale_local_batch_rows", "b200m_group_knn_batch", "b200m_group_match_batch",
           "b200m_group_match_multiscale_batch", "b200m_group_match_multiscale_local_batch", "b200m_batch_partition"]

_lib = None


def load_library():
    """dlopen libb200match.so (built in-tree by lidar_global_registration_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise B200MatchError("libb200match.so is not built (run `python -m lidar_global_registration_b200.build`); "
                             "there is no CPU fallback")
    L = C.CDLL(_LIB_PATH)
    vp, sz, i32, i64, fp = C.c_void_p, C.c_size_t, C.c_int32, C.c_int64, C.c_void_p
    L.b200m_create.argtypes = [C.POINTER(vp), C.c_int]
    L.b200m_destroy.argtypes = [vp]
    L.b200m_destroy.restype = None
    L.b200m_last_error.argtypes = [vp]
    L.b200m_last_error.restype = C.c_char_p
    L.b200m_set_stream.argtypes = [vp, vp]
    L.b200m_sync.argtypes = [vp]
    L.b200m_set_profiling.argtypes = [vp, C.c_int]
    L.b200m_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.b200m_reset_stats.argtypes = [vp]
    L.b200m_upload.argtypes = [vp, C.c_int, fp, sz, sz, C.c_int, i64]
    L.b200m_upload_device.argtypes = [vp, C.c_int, fp, sz, sz, C.c_int, i64]
    L.b200m_knn.argtypes = [vp, C.POINTER(_Params), C.c_int, sz, sz, vp, vp, vp]
    L.b200m_knn_device.argtypes = [vp, C.POINTER(_Params), C.c_int, sz, sz, vp, vp, vp]
    L.b200m_match.argtypes = [vp, C.POINTER(_Params), fp, fp, vp, sz, C.POINTER(sz), C.POINTER(C.c_float)]
    L.b200m_filter_device.argtypes = [vp, C.POINTER(_Params), sz, sz, vp, vp, vp, vp, vp, vp, sz, vp, vp, vp, sz, vp, vp]
    L.b200m_merge_device.argtypes = [vp, C.c_int, C.c_int, sz, vp, vp, vp, vp, vp, vp]
    L.b200m_multiscale_begin.argtypes = [vp, sz, C.c_int, C.c_int]
    L.b200m_multiscale_add.argtypes = [vp, C.POINTER(_Params), C.c_int, C.c_int, vp, vp, sz]
    L.b200m_multiscale_vote.argtypes = [vp, fp, sz, sz, C.c_float, vp, vp, vp]
    L.b200m_multiscale_add_device.argtypes = [vp, C.c_int, sz, vp, vp, vp, vp, vp, sz, i64, sz]
    L.b200m_multiscale_vote_device.argtypes = [vp, fp, sz, C.c_float, vp, vp, vp]
    L.b200m_match_cluster.argtypes = [vp, C.POINTER(_Params), C.c_int, fp, fp, sz, fp, fp, vp, sz, C.POINTER(sz),
                                      C.POINTER(C.c_float)]
    L.b200m_cluster_filter_device.argtypes = [vp, C.POINTER(_Params), C.c_int, C.c_float, sz, sz, vp, vp, vp, vp, vp, fp, fp,
                                              sz, fp, fp, vp, sz, vp, vp]
    L.b200m_knn3d_device.argtypes = [vp, fp, sz, sz, C.c_int, vp]
    L.b200m_mark_referenced_device.argtypes = [vp, C.c_int, vp, vp, sz, i64, vp, sz]
    L.b200m_knn_masked_device.argtypes = [vp, C.POINTER(_Params), C.c_int, sz, sz, vp, vp, vp, vp]
    L.b200m_knn_local.argtypes = [vp, C.POINTER(_Params), C.c_int, fp, fp, sz, C.c_float, vp, vp, vp]
    L.b200m_knn_local_device.argtypes = [vp, C.POINTER(_Params), C.c_int, fp, fp, sz, C.c_float, vp, vp, vp]
    L.b200m_match_multiscale.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Scale), C.c_int, sz, C.c_int, fp, sz, fp, sz, sz,
                                         C.c_float, C.c_float, C.c_int, fp, fp, vp, sz, C.POINTER(sz), C.POINTER(C.c_float)]
    L.b200m_comm_unique_id.argtypes = [vp, sz]
    L.b200m_comm_attach.argtypes = [vp, C.c_int, C.c_int, vp]
    L.b200m_comm_rank.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.b200m_shard_rows.argtypes = [sz, C.c_int, C.c_int, C.POINTER(sz), C.POINTER(sz)]
    L.b200m_upload_replicated.argtypes = [vp, C.c_int, fp, sz, sz, C.c_int]
    L.b200m_match_sharded.argtypes = [vp, C.POINTER(_Params), fp, fp, vp, sz, C.POINTER(sz), C.POINTER(C.c_float)]
    L.b200m_match_sharded_device.argtypes = [vp, C.POINTER(_Params), fp, fp, vp, sz, vp, vp]
    L.b200m_knn_target_sharded_device.argtypes = [vp, C.POINTER(_Params), vp, vp, vp]
    L.b200m_create_multi.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.c_int]
    L.b200m_destroy_multi.argtypes = [vp]
    L.b200m_destroy_multi.restype = None
    L.b200m_group_last_error.argtypes = [vp]
    L.b200m_group_last_error.restype = C.c_char_p
    L.b200m_group_size.argtypes = [vp]
    L.b200m_group_ctx.argtypes = [vp, C.c_int]
    L.b200m_group_ctx.restype = vp
    L.b200m_group_upload.argtypes = [vp, C.c_int, fp, sz, sz, C.c_int]
    L.b200m_group_upload_sharded.argtypes = [vp, C.c_int, fp, sz, sz, C.c_int]
    L.b200m_group_match.argtypes = [vp, C.POINTER(_Params), fp, fp, vp, sz, C.POINTER(sz), C.POINTER(C.c_float)]
    L.b200m_group_knn.argtypes = [vp, C.POINTER(_Params), vp, vp, vp]
    L.b200m_knn_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Pair), C.c_int, sz, C.c_int, vp, vp, vp]
    L.b200m_match_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Pair), C.c_int, sz, C.c_int, fp, fp, vp, sz,
                                    C.POINTER(sz), vp]
    L.b200m_match_multiscale_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_WidePair), C.c_int, sz, C.c_int, sz, C.c_int,
                                               fp, fp, vp, sz, C.POINTER(sz), vp]
    L.b200m_match_multiscale_local_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_WidePair), C.POINTER(_LocalPair), C.c_int, sz,
                                                     C.c_int, sz, C.c_int, C.c_float, fp, fp, vp, sz, C.POINTER(sz), vp]
    L.b200m_knn_batch_device.argtypes = L.b200m_knn_batch.argtypes
    L.b200m_group_knn_batch.argtypes = L.b200m_knn_batch.argtypes
    L.b200m_group_match_batch.argtypes = L.b200m_match_batch.argtypes
    L.b200m_group_match_multiscale_batch.argtypes = L.b200m_match_multiscale_batch.argtypes
    L.b200m_group_match_multiscale_local_batch.argtypes = L.b200m_match_multiscale_local_batch.argtypes
    L.b200m_batch_partition.argtypes = [vp, C.c_int, C.c_int, vp]
    L.b200m_match_batch_device.argtypes = L.b200m_match_batch.argtypes
    L.b200m_match_multiscale_batch_device.argtypes = L.b200m_match_multiscale_batch.argtypes
    L.b200m_match_multiscale_local_batch_device.argtypes = L.b200m_match_multiscale_local_batch.argtypes
    L.b200m_plan_knn_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Pair), C.c_int, sz, C.c_int, vp, vp, vp, C.POINTER(vp)]
    L.b200m_plan_match_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_Pair), C.c_int, sz, C.c_int, vp, vp, vp, sz, vp, vp,
                                         vp, C.POINTER(vp)]
    L.b200m_plan_knn_batch_rows.argtypes = L.b200m_plan_knn_batch.argtypes[:-1] + [vp, vp, C.POINTER(vp)]
    L.b200m_plan_match_batch_rows.argtypes = L.b200m_plan_match_batch.argtypes[:-1] + [vp, vp, C.POINTER(vp)]
    L.b200m_plan_match_multiscale_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_WidePair), C.c_int, sz, C.c_int, sz,
                                                    C.c_int, vp, vp, vp, sz, vp, vp, vp, vp, C.POINTER(vp)]
    L.b200m_plan_match_multiscale_local_batch.argtypes = [vp, C.POINTER(_Params), C.POINTER(_WidePair), C.POINTER(_LocalPair),
                                                          C.c_int, sz, C.c_int, sz, C.c_int, C.c_float, vp, vp, vp, sz, vp, vp,
                                                          vp, vp, C.POINTER(vp)]
    L.b200m_plan_match_multiscale_batch_rows.argtypes = L.b200m_plan_match_multiscale_batch.argtypes[:-1] + [vp, vp, C.POINTER(vp)]
    L.b200m_plan_match_multiscale_local_batch_rows.argtypes = \
        L.b200m_plan_match_multiscale_local_batch.argtypes[:-1] + [vp, vp, C.POINTER(vp)]
    L.b200m_plan_status_error.argtypes = [vp, C.c_uint64]
    L.b200m_plan_status_error.restype = C.c_char_p
    L.b200m_plan_run.argtypes = [vp, vp]
    L.b200m_plan_destroy.argtypes = [vp]
    L.b200m_plan_destroy.restype = None
    L.b200m_plan_last_error.argtypes = [vp]
    L.b200m_plan_last_error.restype = C.c_char_p
    L.b200m_version.restype = C.c_int
    L.b200m_debug_operands.argtypes = [vp, C.c_int, C.c_int, vp, sz, vp, C.POINTER(C.c_float), C.POINTER(i32),
                                       C.POINTER(i64)]
    L.b200m_debug_tc_tile.argtypes = [vp, C.c_int, sz, sz, vp]
    L.b200m_debug_candidate_lists.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64), C.POINTER(i32), vp, vp, vp,
                                              vp]
    _lib = L
    return L


@dataclass
class AlignmentParameters:
    """The fields of the reference's AlignmentParameters read on the matching path
    (include/common.h:135-163) plus the B200-specific knobs."""
    randomness: int = 1                 # k (:147)
    use_bfmatcher: bool = True          # :144 -- both backends map to the same exact GPU search
    bf_block_size: int = 10000          # :145 -- accepted, unused: the GPU streams the whole train set
    distance_thr: float = FLT_MAX       # :139
    ratio_k: int = MATCHING_RATIO_K     # :146
    cluster_k: int = MATCHING_CLUSTER_K  # :146
    matching_id: str = MATCHING_LEFT_TO_RIGHT   # :149
    ratio_thr: float = MATCHING_RATIO_THRESHOLD
    precision: int = PREC_TC_F16
    cand_cap: int = 0
    match_search_radius: float = FLT_MAX   # :160  matchLocal's 3-D gate, used when `guess` is set
    guess: tuple | None = None          # :161  prior pose: 16 floats, row-major (the reference's Eigen::Matrix4f)


def guess_matrix(guess):
    """A guess (16 numbers, row-major, or a 4x4 array) as a float32 [4, 4] array."""
    g = np.asarray(guess, np.float32)
    if g.size != 16:
        raise B200MatchError("guess must have 16 entries (a row-major 4x4 matrix)")
    return g.reshape(4, 4)


def invert_guess(guess):
    """The inverse of a guess, taken in float64 and rounded to float32 (the pose the reverse matchLocal call moves the target
    keypoints by)."""
    return np.linalg.inv(guess_matrix(guess).astype(np.float64)).astype(np.float32)


def transform_keypoints(xyz, guess):
    """Keypoints moved by a guess: x' = ((g00 x + g01 y) + g02 z) + g03 in float32, every product and sum rounded on its
    own -- the order of the C++ shim's matchLocal.  xyz: [n, >= 3]; returns a float32 copy in which only the first three
    columns changed.  A PCL build moves its clouds with transformPointCloudWithNormals instead and passes those."""
    x = np.array(xyz, np.float32, copy=True, ndmin=2)
    if x.ndim != 2 or x.shape[1] < 3:
        raise B200MatchError("keypoint coordinates must be [n, >= 3]")
    g = guess_matrix(guess)
    c = [x[:, 0].copy(), x[:, 1].copy(), x[:, 2].copy()]
    for r in range(3):
        x[:, r] = ((g[r, 0] * c[0] + g[r, 1] * c[1]) + g[r, 2] * c[2]) + g[r, 3]
    return x


def _as_rows(a):
    a = np.asarray(a)
    if a.dtype != np.float32 or a.ndim != 2:
        raise B200MatchError("descriptors must be a 2-D float32 array [n, stride_floats]")
    if a.shape[0] > 1 and (a.strides[1] != 4 or a.strides[0] % 4 != 0 or a.strides[0] < 4 * a.shape[1]):
        a = np.ascontiguousarray(a)
    stride = a.strides[0] if a.shape[0] > 1 else 4 * a.shape[1]
    return a, stride


class Context:
    """One b200m_ctx: one GPU, one stream; calls are serialised (reference call sites are single-threaded)."""

    def __init__(self, device=0):
        self._L = load_library()
        self._h = C.c_void_p()
        if self._L.b200m_create(C.byref(self._h), int(device)) != 0:
            raise B200MatchError(self._L.b200m_last_error(None).decode())
        self.device = int(device)
        self.n = [0, 0]
        self.dim = 0
        self.rank, self.n_ranks = 0, 1

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.b200m_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise B200MatchError(self._L.b200m_last_error(self._h).decode())

    @staticmethod
    def _params(k, mode, ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, precision=PREC_TC_F16, cand_cap=0,
                n_gpus=0, shard=SHARD_QUERY):
        return _Params(int(k), int(mode), float(ratio_thr), float(distance_thr), int(precision), int(cand_cap), int(n_gpus),
                       int(shard))

    # -- plumbing ------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr):
        self._ck(self._L.b200m_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def sync(self):
        self._ck(self._L.b200m_sync(self._h))

    def set_profiling(self, on):
        self._ck(self._L.b200m_set_profiling(self._h, 1 if on else 0))

    def reset_stats(self):
        self._ck(self._L.b200m_reset_stats(self._h))

    def stats(self):
        s = Stats()
        self._ck(self._L.b200m_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # -- upload ---------------------------------------------------------------
    def upload(self, side, rows, dim, index_offset=0):
        """rows: float32 [n, stride_floats] host array (AoS point structs); the first `dim` columns are used."""
        a, stride = _as_rows(rows)
        if dim > a.shape[1]:
            raise B200MatchError("dim exceeds the row length")
        self._keep = getattr(self, "_keep", {})
        self._keep[side] = a
        self._ck(self._L.b200m_upload(self._h, side, a.ctypes.data, a.shape[0], stride, dim, index_offset))
        self.n[side] = a.shape[0]
        self.dim = dim

    def upload_device(self, side, ptr, n, stride_bytes, dim, index_offset=0):
        self._ck(self._L.b200m_upload_device(self._h, side, C.c_void_p(ptr), n, stride_bytes, dim, index_offset))
        self.n[side] = n
        self.dim = dim

    # -- multi-GPU: one process per GPU (SURVEY 8e) ----------------------------------------
    def comm_attach(self, n_ranks, rank, unique_id):
        """ncclCommInitRank on this context's device; `unique_id` = the 128 bytes of comm_unique_id() made on one rank."""
        buf = C.create_string_buffer(bytes(unique_id), UNIQUE_ID_BYTES)
        self._ck(self._L.b200m_comm_attach(self._h, int(n_ranks), int(rank), buf))
        self.rank, self.n_ranks = int(rank), int(n_ranks)

    def upload_replicated(self, side, rows, dim):
        """Collective: every rank passes the same HOST set, copies 1/ranks of it over PCIe; NVLink all-gather; pack."""
        a, stride = _as_rows(rows)
        self._ck(self._L.b200m_upload_replicated(self._h, side, a.ctypes.data, a.shape[0], stride, dim))
        self.n[side] = a.shape[0]
        self.dim = dim

    def match_sharded(self, k, mode, ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, thr_src=None, thr_tgt=None,
                      precision=PREC_TC_F16, cand_cap=0):
        """Collective, query-sharded: returns (this rank's slice of the correspondences, average over ALL source rows)."""
        lo, hi = shard_rows(self.n[0], self.n_ranks, self.rank)
        out = np.empty(max((hi - lo) * (k if mode == MODE_MUTUAL else 1), 1), CORR_DTYPE)
        ts = None if thr_src is None else np.ascontiguousarray(thr_src, np.float32)
        tt = None if thr_tgt is None else np.ascontiguousarray(thr_tgt, np.float32)
        p = self._params(k, mode, ratio_thr, distance_thr, precision, cand_cap)
        n_out, avg = C.c_size_t(0), C.c_float(0)
        self._ck(self._L.b200m_match_sharded(self._h, C.byref(p), None if ts is None else ts.ctypes.data,
                                             None if tt is None else tt.ctypes.data, out.ctypes.data, out.shape[0],
                                             C.byref(n_out), C.byref(avg)))
        return out[:n_out.value], float(avg.value)

    def match_sharded_device(self, k, mode, out_ptr, cap, n_out_ptr, avg_ptr=0, thr_src=0, thr_tgt=0,
                             ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, precision=PREC_TC_F16, cand_cap=0):
        p = self._params(k, mode, ratio_thr, distance_thr, precision, cand_cap)
        v = C.c_void_p
        self._ck(self._L.b200m_match_sharded_device(self._h, C.byref(p), v(thr_src), v(thr_tgt), v(out_ptr), cap, v(n_out_ptr),
                                                    v(avg_ptr)))

    def knn_target_sharded_device(self, k, idx_ptr, dist_ptr, cnt_ptr, precision=PREC_TC_F16, cand_cap=0):
        p = self._params(k, MODE_KNN_ONLY, precision=precision, cand_cap=cand_cap, shard=SHARD_TARGET)
        v = C.c_void_p
        self._ck(self._L.b200m_knn_target_sharded_device(self._h, C.byref(p), v(idx_ptr), v(dist_ptr), v(cnt_ptr)))

    # -- raw k-lists ----------------------------------------------------------
    def knn(self, k, direction=0, row_begin=0, row_end=0, precision=PREC_TC_F16, cand_cap=0):
        nq = self.n[direction]
        re = nq if row_end == 0 else row_end
        rows = max(re - row_begin, 0)
        idx = np.empty((rows, k), np.int32)
        dist = np.empty((rows, k), np.float32)
        cnt = np.empty((rows,), np.int32)
        p = self._params(k, MODE_KNN_ONLY, precision=precision, cand_cap=cand_cap)
        self._ck(self._L.b200m_knn(self._h, C.byref(p), direction, row_begin, re, idx.ctypes.data, dist.ctypes.data,
                                   cnt.ctypes.data))
        return idx, dist, cnt

    def knn_local(self, k, query_xyz, train_xyz, radius, direction=0):
        """matchLocal with a finite match_search_radius: query_xyz are the query keypoints after the guess transform."""
        qx = np.ascontiguousarray(query_xyz, np.float32)
        tx = np.ascontiguousarray(train_xyz, np.float32)
        nq, nt = self.n[direction], self.n[1 - direction]
        if qx.ndim != 2 or tx.ndim != 2 or qx.shape[1] < 3 or qx.shape[1] != tx.shape[1] or qx.shape[0] != nq or tx.shape[0] != nt:
            raise B200MatchError("keypoint coordinates: [n, >= 3] float32, one row per descriptor row, same row length on both sides")
        idx, dist, cnt = np.empty((nq, k), np.int32), np.empty((nq, k), np.float32), np.empty((nq,), np.int32)
        p = self._params(k, MODE_KNN_ONLY)
        self._ck(self._L.b200m_knn_local(self._h, C.byref(p), direction, qx.ctypes.data, tx.ctypes.data, qx.strides[0],
                                         float(radius), idx.ctypes.data, dist.ctypes.data, cnt.ctypes.data))
        return idx, dist, cnt

    def knn_device(self, k, direction, row_begin, row_end, idx_ptr, dist_ptr, cnt_ptr, precision=PREC_TC_F16, cand_cap=0):
        p = self._params(k, MODE_KNN_ONLY, precision=precision, cand_cap=cand_cap)
        self._ck(self._L.b200m_knn_device(self._h, C.byref(p), direction, row_begin, row_end, C.c_void_p(idx_ptr),
                                          C.c_void_p(dist_ptr), C.c_void_p(cnt_ptr)))

    def knn_masked_device(self, k, direction, row_begin, row_end, flags_ptr, idx_ptr, dist_ptr, cnt_ptr, precision=PREC_TC_F16,
                          cand_cap=0):
        p = self._params(k, MODE_KNN_ONLY, precision=precision, cand_cap=cand_cap)
        v = C.c_void_p
        self._ck(self._L.b200m_knn_masked_device(self._h, C.byref(p), direction, row_begin, row_end, v(flags_ptr), v(idx_ptr),
                                                 v(dist_ptr), v(cnt_ptr)))

    def mark_referenced_device(self, k, fidx_ptr, fcnt_ptr, n_rows, index_offset, flags_ptr, n_flags):
        v = C.c_void_p
        self._ck(self._L.b200m_mark_referenced_device(self._h, k, v(fidx_ptr), v(fcnt_ptr), n_rows, index_offset, v(flags_ptr),
                                                      n_flags))

    # -- batches: many (source, target) pairs in one call -------------------------------------
    @staticmethod
    def _pairs(pairs, dim):
        """-> (the contiguous float32 arrays to keep alive, b200m_pair array, stride_bytes, source row counts)."""
        keep, width = [], None
        arr = (_Pair * max(len(pairs), 1))()
        for i, (s, t) in enumerate(pairs):
            s, t = np.ascontiguousarray(s, np.float32), np.ascontiguousarray(t, np.float32)
            if s.ndim != 2 or t.ndim != 2 or s.shape[1] != t.shape[1] or (width is not None and s.shape[1] != width):
                raise B200MatchError("batch: every set must be a 2-D float32 array [n, stride_floats] of one row length")
            width = s.shape[1]
            keep += [s, t]
            arr[i] = _Pair(s.ctypes.data if s.shape[0] else None, s.shape[0], t.ctypes.data if t.shape[0] else None, t.shape[0])
        if width is not None and dim > width:
            raise B200MatchError("dim exceeds the row length")
        return keep, arr, 4 * (width or dim), [int(s.shape[0]) for s, _ in pairs]

    def _batch_call(self, name):
        # the host batch calls: b200m_<name> on this context (Group: b200m_group_<name>)
        return getattr(self._L, "b200m_" + name)

    def _batch_sides(self, pairs):
        # what the library's two sides hold after a batch call: every set padded to a multiple of 256 rows
        self._batch_rows([(len(s), len(t)) for s, t in pairs])

    def _batch_rows(self, counts):
        self.n = [sum(-(-int(c[s]) // 256) * 256 for c in counts) for s in (0, 1)]

    def knn_batch(self, k, pairs, dim, precision=PREC_TC_F16, cand_cap=0):
        """b200m_knn_batch: `pairs` = [(source rows, target rows), ...] (float32 [n, stride_floats], one row length).
        Returns one (idx, dist, count) per pair, each equal to upload + knn(k, 0) on that pair alone.  Replaces the sets
        uploaded before."""
        keep, arr, stride, ns = self._pairs(pairs, dim)
        total = sum(ns)
        idx = np.empty((total, k), np.int32)
        dist = np.empty((total, k), np.float32)
        cnt = np.empty((total,), np.int32)
        p = self._params(k, MODE_KNN_ONLY, precision=precision, cand_cap=cand_cap)
        self._ck(self._batch_call("knn_batch")(self._h, C.byref(p), arr, len(pairs), stride, dim, idx.ctypes.data, dist.ctypes.data,
                                               cnt.ctypes.data))
        self._batch_sides(pairs)
        off = np.concatenate([[0], np.cumsum(ns)]).astype(np.int64)
        return [(idx[a:b], dist[a:b], cnt[a:b]) for a, b in zip(off[:-1], off[1:])]

    def match_batch(self, k, mode, pairs, dim, ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, thr_src=None,
                    thr_tgt=None, precision=PREC_TC_F16, cand_cap=0):
        """b200m_match_batch: returns one (correspondences as CORR_DTYPE array, average first-NN distance) per pair, each
        equal to upload + match on that pair alone (pair-local indices).  thr_src / thr_tgt: None or one threshold array per
        pair.  Replaces the sets uploaded before."""
        keep, arr, stride, ns = self._pairs(pairs, dim)
        if (thr_src is None) != (thr_tgt is None):
            raise B200MatchError("give both threshold lists or neither")
        ts = tt = None
        if thr_src is not None:
            if len(thr_src) != len(pairs) or len(thr_tgt) != len(pairs):
                raise B200MatchError("one threshold array per pair and side")
            for i, (s, t) in enumerate(pairs):
                if len(thr_src[i]) != len(s) or len(thr_tgt[i]) != len(t):
                    raise B200MatchError("pair %d: threshold array length != number of rows" % i)
            ts = np.concatenate([np.asarray(a, np.float32).ravel() for a in thr_src] + [np.zeros(1, np.float32)])
            tt = np.concatenate([np.asarray(a, np.float32).ravel() for a in thr_tgt] + [np.zeros(1, np.float32)])
        kk = k if mode == MODE_MUTUAL else 1
        out = np.empty(max(sum(ns) * kk, 1), CORR_DTYPE)
        offsets = np.zeros(len(pairs) + 1, np.uint64)
        avg = np.empty(max(len(pairs), 1), np.float32)
        p = self._params(k, mode, ratio_thr, distance_thr, precision, cand_cap)
        self._ck(self._batch_call("match_batch")(self._h, C.byref(p), arr, len(pairs), stride, dim,
                                                 None if ts is None else ts.ctypes.data, None if tt is None else tt.ctypes.data,
                                                 out.ctypes.data, out.shape[0], offsets.ctypes.data_as(C.POINTER(C.c_size_t)),
                                                 avg.ctypes.data))
        self._batch_sides(pairs)
        return [(out[int(offsets[i]):int(offsets[i + 1])], float(avg[i])) for i in range(len(pairs))]

    # -- device-resident batches: every data pointer below is a device pointer on this context's device --------------
    @staticmethod
    def _device_pairs(pairs):
        """[(src_ptr, n_src, tgt_ptr, n_tgt), ...] -> b200m_pair array."""
        arr = (_Pair * max(len(pairs), 1))()
        for i, (s, ns, t, nt) in enumerate(pairs):
            arr[i] = _Pair(s or None, int(ns), t or None, int(nt))
        return arr

    def knn_batch_device(self, k, pairs, stride_bytes, dim, idx_ptr, dist_ptr, cnt_ptr, precision=PREC_TC_F16, cand_cap=0):
        """b200m_knn_batch_device: `pairs` = [(src_ptr, n_src, tgt_ptr, n_tgt), ...]; the k-lists go to the device arrays
        idx [sum n_src][k], dist, cnt.  Replaces the sets uploaded before."""
        p = self._params(k, MODE_KNN_ONLY, precision=precision, cand_cap=cand_cap)
        v = C.c_void_p
        self._ck(self._L.b200m_knn_batch_device(self._h, C.byref(p), self._device_pairs(pairs), len(pairs), stride_bytes, dim,
                                                v(idx_ptr), v(dist_ptr), v(cnt_ptr)))
        self._batch_rows([(ns, nt) for _, ns, _, nt in pairs])

    def match_batch_device(self, k, mode, pairs, stride_bytes, dim, out_ptr, cap, thr_src=0, thr_tgt=0,
                           ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, precision=PREC_TC_F16, cand_cap=0):
        """b200m_match_batch_device: `pairs` as knn_batch_device's; records go to the device buffer out_ptr (`cap` records),
        thr_src / thr_tgt are device pointers to the concatenated thresholds or 0.  -> (offsets uint64 [n_pairs + 1],
        averages float32 [n_pairs]) on the host."""
        offsets = np.zeros(len(pairs) + 1, np.uint64)
        avg = np.empty(max(len(pairs), 1), np.float32)
        p = self._params(k, mode, ratio_thr, distance_thr, precision, cand_cap)
        v = C.c_void_p
        self._ck(self._L.b200m_match_batch_device(self._h, C.byref(p), self._device_pairs(pairs), len(pairs), stride_bytes, dim,
                                                  v(thr_src), v(thr_tgt), v(out_ptr), cap,
                                                  offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data))
        self._batch_rows([(ns, nt) for _, ns, _, nt in pairs])
        return offsets, avg[:len(pairs)]

    def match_wide_batch_device(self, k, mode, pairs, stride_bytes, dim, xyz_stride_bytes, out_ptr, cap,
                                cluster_k=MATCHING_CLUSTER_K, distance_thr=FLT_MAX, thr_src=0, thr_tgt=0, precision=PREC_TC_F16,
                                cand_cap=0):
        """b200m_match_multiscale_batch_device.  Each entry of `pairs` is a dict: scales = [(src_ptr, n_src, src_map_ptr,
        tgt_ptr, n_tgt, tgt_map_ptr), ...] (map 0: identity), src_kps_xyz / tgt_kps_xyz (pointers), n_src_kps, n_tgt_kps,
        iss_radius_src, iss_radius_tgt.  -> (offsets, averages) as match_batch_device's."""
        return self._wide_batch_device(k, mode, pairs, None, stride_bytes, dim, xyz_stride_bytes, out_ptr, cap, cluster_k,
                                       distance_thr, thr_src, thr_tgt, precision, cand_cap)

    def match_wide_local_batch_device(self, k, mode, pairs, match_search_radius, stride_bytes, dim, xyz_stride_bytes, out_ptr,
                                      cap, cluster_k=MATCHING_CLUSTER_K, distance_thr=FLT_MAX, thr_src=0, thr_tgt=0):
        """b200m_match_multiscale_local_batch_device: match_wide_batch_device's dicts plus the pointers src_kps_moved and
        tgt_kps_moved (0 allowed in ONE_SIDED mode)."""
        return self._wide_batch_device(k, mode, pairs, float(match_search_radius), stride_bytes, dim, xyz_stride_bytes, out_ptr,
                                       cap, cluster_k, distance_thr, thr_src, thr_tgt, PREC_TC_F16, 0)

    @staticmethod
    def _wide_device_pairs(pairs, gated):
        """match_wide_batch_device's dicts -> (b200m_wide_pair array, b200m_local_pair array, the scale arrays they point to)."""
        keep, arr = [], (_WidePair * max(len(pairs), 1))()
        locs = (_LocalPair * max(len(pairs), 1))()
        for i, f in enumerate(pairs):
            sc = (_Scale * max(len(f["scales"]), 1))()
            for s, (a, na, ma, b, nb, mb) in enumerate(f["scales"]):
                sc[s] = _Scale(a or None, int(na), ma or None, b or None, int(nb), mb or None)
            keep.append(sc)
            arr[i] = _WidePair(C.cast(sc, C.c_void_p), len(f["scales"]), f.get("src_kps_xyz") or None, int(f["n_src_kps"]),
                               f.get("tgt_kps_xyz") or None, int(f["n_tgt_kps"]), float(f["iss_radius_src"]),
                               float(f["iss_radius_tgt"]))
            if gated:
                locs[i] = _LocalPair(f.get("src_kps_moved") or None, f.get("tgt_kps_moved") or None)
        return arr, locs, keep

    def _wide_batch_device(self, k, mode, pairs, radius, stride_bytes, dim, xyz_stride_bytes, out_ptr, cap, cluster_k,
                           distance_thr, thr_src, thr_tgt, precision, cand_cap):
        arr, locs, keep = self._wide_device_pairs(pairs, radius is not None)
        offsets = np.zeros(len(pairs) + 1, np.uint64)
        avg = np.empty(max(len(pairs), 1), np.float32)
        p = self._params(k, mode, distance_thr=distance_thr, precision=precision, cand_cap=cand_cap)
        v = C.c_void_p
        tail = (v(thr_src), v(thr_tgt), v(out_ptr), cap, offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data)
        if radius is None:
            self._ck(self._L.b200m_match_multiscale_batch_device(self._h, C.byref(p), arr, len(pairs), stride_bytes, dim,
                                                                 xyz_stride_bytes, int(cluster_k), *tail))
        else:
            self._ck(self._L.b200m_match_multiscale_local_batch_device(self._h, C.byref(p), arr, locs, len(pairs), stride_bytes, dim,
                                                                       xyz_stride_bytes, int(cluster_k), radius, *tail))
        # what the library's two sides hold afterwards: the last scale's sets of every pair, each padded to 256 rows
        n_last = max((len(f["scales"]) for f in pairs if f["n_src_kps"]), default=0)
        if n_last:
            self._batch_rows([(f["scales"][n_last - 1][1], f["scales"][n_last - 1][4])
                              if f["n_src_kps"] and len(f["scales"]) >= n_last else (0, 0) for f in pairs])
        return offsets, avg[:len(pairs)]

    # -- whole matcher call ----------------------------------------------------
    def match(self, k, mode, ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, thr_src=None, thr_tgt=None,
              precision=PREC_TC_F16, cand_cap=0, out=None):
        """Returns (correspondences as CORR_DTYPE array, average first-NN distance)."""
        nq = self.n[0]
        kk = k if mode == MODE_MUTUAL else 1
        if out is None:
            out = np.empty(max(nq * kk, 1), CORR_DTYPE)
        ts = None if thr_src is None else np.ascontiguousarray(thr_src, np.float32)
        tt = None if thr_tgt is None else np.ascontiguousarray(thr_tgt, np.float32)
        if ts is not None and ts.shape[0] != nq:
            raise B200MatchError("thr_src length != number of source rows")
        if tt is not None and tt.shape[0] != self.n[1]:
            raise B200MatchError("thr_tgt length != number of target rows")
        p = self._params(k, mode, ratio_thr, distance_thr, precision, cand_cap)
        n_out = C.c_size_t(0)
        avg = C.c_float(0)
        self._ck(self._L.b200m_match(self._h, C.byref(p), None if ts is None else ts.ctypes.data,
                                     None if tt is None else tt.ctypes.data, out.ctypes.data, out.shape[0],
                                     C.byref(n_out), C.byref(avg)))
        return out[:n_out.value], float(avg.value)

    def filter_device(self, k, mode, row_begin, row_end, fidx, fdist, fcnt, ridx, rdist, rcnt, n_rev_rows, out_ptr, cap,
                      n_out_ptr, avg_ptr=0, thr_src=0, thr_tgt=0, ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX):
        p = self._params(k, mode, ratio_thr, distance_thr)
        v = C.c_void_p
        self._ck(self._L.b200m_filter_device(self._h, C.byref(p), row_begin, row_end, v(fidx), v(fdist), v(fcnt), v(ridx),
                                             v(rdist), v(rcnt), n_rev_rows, v(thr_src), v(thr_tgt), v(out_ptr), cap,
                                             v(n_out_ptr), v(avg_ptr)))

    def merge_device(self, k, n_lists, nq, idx_in, dist_in, cnt_in, idx, dist, cnt):
        v = C.c_void_p
        self._ck(self._L.b200m_merge_device(self._h, k, n_lists, nq, v(idx_in), v(dist_in), v(cnt_in), v(idx), v(dist),
                                            v(cnt)))

    # -- ClusterMatcher::match_impl (include/matching.h:492-517) ---------------------------
    def match_cluster(self, k, cluster_k, src_kps_xyz, tgt_kps_xyz, distance_thr=FLT_MAX, thr_src=None, thr_tgt=None,
                      precision=PREC_TC_F16, out=None):
        """Returns (correspondences as CORR_DTYPE array, average first-NN distance)."""
        nq, nt = self.n
        sx = np.ascontiguousarray(src_kps_xyz, np.float32)
        tx = np.ascontiguousarray(tgt_kps_xyz, np.float32)
        if sx.ndim != 2 or tx.ndim != 2 or sx.shape[1] < 3 or sx.shape[1] != tx.shape[1]:
            raise B200MatchError("keypoint coordinates must be [n, >= 3] float32 with the same row length on both sides")
        if sx.shape[0] != nq or tx.shape[0] != nt:
            raise B200MatchError("one keypoint per descriptor row is needed on both sides")
        if out is None:
            out = np.empty(max(nq * k, 1), CORR_DTYPE)
        ts = None if thr_src is None else np.ascontiguousarray(thr_src, np.float32)
        tt = None if thr_tgt is None else np.ascontiguousarray(thr_tgt, np.float32)
        p = self._params(k, MODE_CLUSTER, distance_thr=distance_thr, precision=precision)
        n_out, avg = C.c_size_t(0), C.c_float(0)
        self._ck(self._L.b200m_match_cluster(self._h, C.byref(p), int(cluster_k), sx.ctypes.data, tx.ctypes.data, sx.strides[0],
                                             None if ts is None else ts.ctypes.data, None if tt is None else tt.ctypes.data,
                                             out.ctypes.data, out.shape[0], C.byref(n_out), C.byref(avg)))
        return out[:n_out.value], float(avg.value)

    # -- the matcher classes at the wide seam (match_impl: match_multiscale both ways + filter) ----
    def match_wide(self, k, mode, src_scales, tgt_scales, src_kps_xyz, tgt_kps_xyz, iss_radius_src, iss_radius_tgt, dim=None,
                   cluster_k=MATCHING_CLUSTER_K, distance_thr=FLT_MAX, thr_src=None, thr_tgt=None, precision=PREC_TC_F16,
                   cand_cap=0):
        """OneSided / LeftToRight / ClusterMatcher::match_impl (include/matching.h:395-411, :428-453, :492-517) over
        precomputed per-scale descriptors: `src_scales` / `tgt_scales` are lists, one entry per common scale, of
        (features [n_s, >= dim] float32, kps_indices_multiscale [n_s] int32 or None).  Returns (correspondences over
        keypoint ids, average first-NN distance of the voted forward lists)."""
        if len(src_scales) != len(tgt_scales) or not src_scales:
            raise B200MatchError("match_wide: need the same, non-zero number of scales on both sides")
        sx = np.ascontiguousarray(src_kps_xyz, np.float32)
        tx = np.ascontiguousarray(tgt_kps_xyz, np.float32)
        if sx.ndim != 2 or tx.ndim != 2 or sx.shape[1] < 3 or sx.shape[1] != tx.shape[1]:
            raise B200MatchError("keypoint coordinates must be [n, >= 3] float32 with the same row length on both sides")
        keep, arr, width = self._scales(src_scales, tgt_scales)
        d = int(dim or width)
        if d > width:
            raise B200MatchError("dim exceeds the row length")
        ts = None if thr_src is None else np.ascontiguousarray(thr_src, np.float32)
        tt = None if thr_tgt is None else np.ascontiguousarray(thr_tgt, np.float32)
        if (ts is not None and ts.shape[0] != sx.shape[0]) or (tt is not None and tt.shape[0] != tx.shape[0]):
            raise B200MatchError("threshold arrays must have one entry per keypoint")
        out = np.empty(max(sx.shape[0], 1), CORR_DTYPE)
        p = self._params(k, mode, distance_thr=distance_thr, precision=precision, cand_cap=cand_cap)
        n_out, avg = C.c_size_t(0), C.c_float(0)
        self._ck(self._L.b200m_match_multiscale(
            self._h, C.byref(p), arr, len(src_scales), width * 4, d, sx.ctypes.data, sx.shape[0], tx.ctypes.data, tx.shape[0],
            sx.strides[0] if sx.shape[0] > 1 else 4 * sx.shape[1], float(iss_radius_src), float(iss_radius_tgt), int(cluster_k),
            None if ts is None else ts.ctypes.data, None if tt is None else tt.ctypes.data, out.ctypes.data, out.shape[0],
            C.byref(n_out), C.byref(avg)))
        return out[:n_out.value], float(avg.value)

    @staticmethod
    def _scales(src_scales, tgt_scales, width=None):
        """-> (the arrays to keep alive, b200m_scale array, descriptor row length in floats or `width` if no scale)."""
        if len(src_scales) != len(tgt_scales):
            raise B200MatchError("match_wide: need the same number of scales on both sides")
        keep, arr = [], (_Scale * max(len(src_scales), 1))()
        for s, ((sf, smap), (tf, tmap)) in enumerate(zip(src_scales, tgt_scales)):
            sf = np.ascontiguousarray(sf, np.float32)
            tf = np.ascontiguousarray(tf, np.float32)
            if sf.ndim != 2 or tf.ndim != 2 or sf.shape[1] != tf.shape[1] or (width is not None and sf.shape[1] != width):
                raise B200MatchError("match_wide: every scale's descriptor rows must have the same length on both sides")
            width = sf.shape[1]
            sm = None if smap is None else np.ascontiguousarray(smap, np.int32)
            tm = None if tmap is None else np.ascontiguousarray(tmap, np.int32)
            if (sm is not None and sm.shape[0] != sf.shape[0]) or (tm is not None and tm.shape[0] != tf.shape[0]):
                raise B200MatchError("match_wide: index map length != number of descriptor rows of the scale")
            keep += [sf, tf, sm, tm]
            arr[s] = _Scale(sf.ctypes.data if sf.shape[0] else None, sf.shape[0], None if sm is None else sm.ctypes.data,
                            tf.ctypes.data if tf.shape[0] else None, tf.shape[0], None if tm is None else tm.ctypes.data)
        return keep, arr, width

    _WIDE_FIELDS = ("src_scales", "tgt_scales", "src_kps_xyz", "tgt_kps_xyz", "iss_radius_src", "iss_radius_tgt")

    def match_wide_batch(self, k, mode, pairs, dim=None, cluster_k=MATCHING_CLUSTER_K, distance_thr=FLT_MAX, thr_src=None,
                         thr_tgt=None, precision=PREC_TC_F16, cand_cap=0):
        """b200m_match_multiscale_batch: match_wide of many (source, target) cloud pairs in one call.  Each entry of `pairs`
        has match_wide's fields -- a dict with the keys src_scales, tgt_scales, src_kps_xyz, tgt_kps_xyz, iss_radius_src,
        iss_radius_tgt, or a sequence in that order.  Pairs may have different numbers of scales (none too); in ONE_SIDED mode
        src_kps_xyz may be None when the dict gives n_src_kps.  thr_src / thr_tgt: None or one per-keypoint threshold array
        per pair.  Returns one (correspondences over pair-local keypoint ids, average) per pair, each equal to match_wide on
        that pair alone.  Replaces the sets uploaded before."""
        return self._wide_batch(k, mode, pairs, None, dim, cluster_k, distance_thr, thr_src, thr_tgt, precision, cand_cap)

    def match_wide_local_batch(self, k, mode, pairs, match_search_radius, dim=None, cluster_k=MATCHING_CLUSTER_K,
                               distance_thr=FLT_MAX, thr_src=None, thr_tgt=None):
        """b200m_match_multiscale_local_batch: match_wide_batch with AlignmentParameters::guess set -- every scale's kNN is
        matchLocal's, gated at match_search_radius around the MOVED query keypoints.  Each dict of `pairs` has
        match_wide_batch's keys plus src_kps_moved (the source keypoints moved by the pair's guess, e.g. by
        transform_keypoints) and tgt_kps_moved (the target keypoints moved by the guess's inverse; may be None in ONE_SIDED
        mode), with the rows and row length of the unmoved coordinates.  Replaces the sets uploaded before."""
        return self._wide_batch(k, mode, pairs, float(match_search_radius), dim, cluster_k, distance_thr, thr_src, thr_tgt,
                                PREC_TC_F16, 0)

    def _wide_batch(self, k, mode, pairs, radius, dim, cluster_k, distance_thr, thr_src, thr_tgt, precision, cand_cap):
        # radius None: b200m_match_multiscale_batch, else b200m_match_multiscale_local_batch
        if (thr_src is None) != (thr_tgt is None):
            raise B200MatchError("give both threshold lists or neither")
        keep, arr = [], (_WidePair * max(len(pairs), 1))()
        locs = (_LocalPair * max(len(pairs), 1))()
        width = xyz_width = None
        n_kps, fs = [], [dict(pr) if isinstance(pr, dict) else dict(zip(self._WIDE_FIELDS, pr)) for pr in pairs]

        def coords(i, x):
            if x is None:
                return None
            nonlocal xyz_width
            x = np.ascontiguousarray(x, np.float32)
            if x.ndim != 2 or x.shape[1] < 3 or (xyz_width is not None and x.shape[1] != xyz_width):
                raise B200MatchError("pair %d: keypoint coordinates must be [n, >= 3] float32, one row length in the batch" % i)
            xyz_width = x.shape[1]
            return x

        for i, f in enumerate(fs):
            k_keep, sc, width = self._scales(f["src_scales"], f["tgt_scales"], width)
            xs = [coords(i, f.get(side)) for side in ("src_kps_xyz", "tgt_kps_xyz")]
            if xs[1] is None:
                raise B200MatchError("pair %d: tgt_kps_xyz is needed" % i)
            ns = xs[0].shape[0] if xs[0] is not None else int(f.get("n_src_kps", 0))
            n_kps.append((ns, xs[1].shape[0]))
            keep += [k_keep, sc, xs]
            arr[i] = _WidePair(C.cast(sc, C.c_void_p), len(f["src_scales"]), None if xs[0] is None or not ns else xs[0].ctypes.data, ns,
                               xs[1].ctypes.data if xs[1].shape[0] else None, xs[1].shape[0], float(f["iss_radius_src"]),
                               float(f["iss_radius_tgt"]))
            if radius is not None:
                ms = [coords(i, f.get(side)) for side in ("src_kps_moved", "tgt_kps_moved")]
                for m, n in zip(ms, n_kps[-1]):
                    if m is not None and m.shape[0] != n:
                        raise B200MatchError("pair %d: moved keypoints must have the rows of the unmoved ones" % i)
                keep.append(ms)
                locs[i] = _LocalPair(*[None if m is None or not m.shape[0] else m.ctypes.data for m in ms])
        width = width or int(dim or 1)
        d = int(dim or width)
        if d > width:
            raise B200MatchError("dim exceeds the row length")
        ts = tt = None
        if thr_src is not None:
            if len(thr_src) != len(pairs) or len(thr_tgt) != len(pairs):
                raise B200MatchError("one threshold array per pair and side")
            for i, (ns, nt) in enumerate(n_kps):
                if len(thr_src[i]) != ns or len(thr_tgt[i]) != nt:
                    raise B200MatchError("pair %d: threshold arrays must have one entry per keypoint" % i)
            ts = np.concatenate([np.asarray(a, np.float32).ravel() for a in thr_src] + [np.zeros(1, np.float32)])
            tt = np.concatenate([np.asarray(a, np.float32).ravel() for a in thr_tgt] + [np.zeros(1, np.float32)])
        out = np.empty(max(sum(ns for ns, _ in n_kps), 1), CORR_DTYPE)
        offsets = np.zeros(len(pairs) + 1, np.uint64)
        avg = np.empty(max(len(pairs), 1), np.float32)
        p = self._params(k, mode, distance_thr=distance_thr, precision=precision, cand_cap=cand_cap)
        tail = (None if ts is None else ts.ctypes.data, None if tt is None else tt.ctypes.data, out.ctypes.data, out.shape[0],
                offsets.ctypes.data_as(C.POINTER(C.c_size_t)), avg.ctypes.data)
        if radius is None:
            self._ck(self._batch_call("match_multiscale_batch")(self._h, C.byref(p), arr, len(pairs), width * 4, d,
                                                                4 * (xyz_width or 4), int(cluster_k), *tail))
        else:
            self._ck(self._batch_call("match_multiscale_local_batch")(self._h, C.byref(p), arr, locs, len(pairs), width * 4, d,
                                                                      4 * (xyz_width or 4), int(cluster_k), radius, *tail))
        # what the library's two sides hold afterwards: the last scale's sets of every pair, each padded to 256 rows
        n_last = max((len(f["src_scales"]) for f, (ns, _) in zip(fs, n_kps) if ns), default=0)
        if n_last:
            self._batch_sides([(f["src_scales"][n_last - 1][0], f["tgt_scales"][n_last - 1][0])
                               if ns and len(f["src_scales"]) >= n_last else ((), ()) for f, (ns, _) in zip(fs, n_kps)])
        return [(out[int(offsets[i]):int(offsets[i + 1])], float(avg[i])) for i in range(len(pairs))]

    # -- multi-scale merge + spatial vote (match_multiscale, include/matching.h:264-354) ----
    def multiscale_begin(self, n_query_kps, n_scales, k):
        self._ms = (int(n_query_kps), int(k))
        self._ck(self._L.b200m_multiscale_begin(self._h, n_query_kps, n_scales, k))

    def multiscale_add(self, scale, direction=0, query_map=None, train_map=None, n_train_kps=None, precision=PREC_TC_F16):
        """kNN of the currently uploaded sides (this scale's descriptors) filed under the scale's index maps."""
        qm = None if query_map is None else np.ascontiguousarray(query_map, np.int32)
        tm = None if train_map is None else np.ascontiguousarray(train_map, np.int32)
        if qm is not None and qm.shape[0] != self.n[direction]:
            raise B200MatchError("query_map length != number of query rows of this scale")
        if tm is not None and tm.shape[0] != self.n[1 - direction]:
            raise B200MatchError("train_map length != number of train rows of this scale")
        if n_train_kps is None:
            n_train_kps = self.n[1 - direction] if tm is None else int(tm.max()) + 1 if tm.size else 0
        p = self._params(self._ms[1], MODE_KNN_ONLY, precision=precision)
        self._ck(self._L.b200m_multiscale_add(self._h, C.byref(p), direction, scale, None if qm is None else qm.ctypes.data,
                                              None if tm is None else tm.ctypes.data, n_train_kps))

    def multiscale_vote(self, train_xyz, iss_radius):
        """-> (match index [n_query_kps] (-1: none), descriptor distance, count 0/1)."""
        xyz = np.ascontiguousarray(train_xyz, np.float32)
        if xyz.ndim != 2 or xyz.shape[1] < 3:
            raise B200MatchError("train_xyz must be [n_train_kps, >= 3] float32 (pcl::PointXYZ rows)")
        nq = self._ms[0]
        idx, dist, cnt = np.empty(nq, np.int32), np.empty(nq, np.float32), np.empty(nq, np.int32)
        self._ck(self._L.b200m_multiscale_vote(self._h, xyz.ctypes.data, xyz.shape[0], xyz.strides[0], float(iss_radius),
                                               idx.ctypes.data, dist.ctypes.data, cnt.ctypes.data))
        return idx, dist, cnt

    # -- test hooks -------------------------------------------------------------
    def debug_operands(self, side, as_query):
        kp, n_pad, scale = C.c_int32(0), C.c_int64(0), C.c_float(0)
        self._ck(self._L.b200m_debug_operands(self._h, side, int(as_query), None, 0, None, C.byref(scale), C.byref(kp),
                                              C.byref(n_pad)))
        ops = np.empty((n_pad.value, kp.value), np.float16)
        norm = np.empty((n_pad.value,), np.float32)
        self._ck(self._L.b200m_debug_operands(self._h, side, int(as_query), ops.ctypes.data, ops.size, norm.ctypes.data,
                                              C.byref(scale), C.byref(kp), C.byref(n_pad)))
        return ops, norm, float(scale.value)

    def debug_tc_tile(self, direction, q_row0, t_tile):
        out = np.empty((128, 256), np.float32)
        self._ck(self._L.b200m_debug_tc_tile(self._h, direction, q_row0, t_tile, out.ctypes.data))
        return out

    def debug_candidate_lists(self):
        """The last candidate launch's lists: dict kind, cap, cnt [n_lists][n_rows], idx [n_lists][n_rows][cap] and, for
        kind 1 / 2, val [n_lists][n_rows][cap] and thr [n_lists][n_rows] (None for kind 0).  debug_tc_tile overwrites them."""
        n_lists, cap, kind, n_rows = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int64(0)
        self._ck(self._L.b200m_debug_candidate_lists(self._h, C.byref(n_lists), C.byref(cap), C.byref(n_rows), C.byref(kind),
                                                     None, None, None, None))
        shape = (n_lists.value, n_rows.value)
        cnt = np.empty(shape, np.int32)
        idx = np.empty(shape + (cap.value,), np.int32)
        val = np.empty(shape + (cap.value,), np.float32) if kind.value else None
        thr = np.empty(shape, np.float32) if kind.value else None
        ptr = lambda a: None if a is None else a.ctypes.data
        self._ck(self._L.b200m_debug_candidate_lists(self._h, C.byref(n_lists), C.byref(cap), C.byref(n_rows), C.byref(kind),
                                                     ptr(cnt), ptr(idx), ptr(val), ptr(thr)))
        return {"kind": kind.value, "cap": cap.value, "cnt": cnt, "idx": idx, "val": val, "thr": thr}


def comm_unique_id():
    """128 bytes naming a new NCCL communicator (make it on one rank, hand it to all: Context.comm_attach)."""
    L = load_library()
    buf = C.create_string_buffer(UNIQUE_ID_BYTES)
    if L.b200m_comm_unique_id(buf, UNIQUE_ID_BYTES) != 0:
        raise B200MatchError(L.b200m_last_error(None).decode())
    return buf.raw


def shard_rows(n, n_ranks, rank):
    """The library's row partition: rank r owns [r*R, min(n, (r+1)*R)), R = ceil(n / ranks) (pure host code)."""
    L = load_library()
    lo, hi = C.c_size_t(0), C.c_size_t(0)
    if L.b200m_shard_rows(int(n), int(n_ranks), int(rank), C.byref(lo), C.byref(hi)) != 0:
        raise B200MatchError("shard_rows: bad rank")
    return lo.value, hi.value


class Group:
    """b200m_create_multi: ONE process, one context + one host thread per device inside the library; whole host arrays in
    and out -- the shape of the reference's single FeatureBasedMatcher::match() call (src/correspondence_search.cpp:14-15)."""

    def __init__(self, devices):
        self._L = load_library()
        self._h = C.c_void_p()
        ids = (C.c_int * len(devices))(*[int(d) for d in devices])
        if self._L.b200m_create_multi(C.byref(self._h), ids, len(devices)) != 0:
            raise B200MatchError(self._L.b200m_group_last_error(None).decode())
        self.devices = list(devices)
        self.n = [0, 0]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.b200m_destroy_multi(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise B200MatchError(self._L.b200m_group_last_error(self._h).decode())

    def upload(self, side, rows, dim, sharded=False):
        a, stride = _as_rows(rows)
        self._keep = getattr(self, "_keep", {})
        self._keep[side] = a
        fn = self._L.b200m_group_upload_sharded if sharded else self._L.b200m_group_upload
        self._ck(fn(self._h, side, a.ctypes.data, a.shape[0], stride, dim))
        self.n[side] = a.shape[0]

    def _check_uploaded(self):
        # the library sizes the whole-problem calls from what device 0 holds; after a batch that is not what self.n says
        if None in self.n:
            raise B200MatchError("Group: a batch call replaced the uploaded sets; upload both sides again first")

    def match(self, k, mode, ratio_thr=MATCHING_RATIO_THRESHOLD, distance_thr=FLT_MAX, thr_src=None, thr_tgt=None,
              precision=PREC_TC_F16):
        self._check_uploaded()
        out = np.empty(max(self.n[0] * (k if mode == MODE_MUTUAL else 1), 1), CORR_DTYPE)
        ts = None if thr_src is None else np.ascontiguousarray(thr_src, np.float32)
        tt = None if thr_tgt is None else np.ascontiguousarray(thr_tgt, np.float32)
        p = Context._params(k, mode, ratio_thr, distance_thr, precision)
        n_out, avg = C.c_size_t(0), C.c_float(0)
        self._ck(self._L.b200m_group_match(self._h, C.byref(p), None if ts is None else ts.ctypes.data,
                                           None if tt is None else tt.ctypes.data, out.ctypes.data, out.shape[0],
                                           C.byref(n_out), C.byref(avg)))
        return out[:n_out.value], float(avg.value)

    def knn(self, k, shard=SHARD_QUERY, precision=PREC_TC_F16):
        self._check_uploaded()
        nq = self.n[0]
        idx, dist, cnt = np.empty((nq, k), np.int32), np.empty((nq, k), np.float32), np.empty((nq,), np.int32)
        p = Context._params(k, MODE_KNN_ONLY, precision=precision, shard=shard)
        self._ck(self._L.b200m_group_knn(self._h, C.byref(p), idx.ctypes.data, dist.ctypes.data, cnt.ctypes.data))
        return idx, dist, cnt

    # -- the host batch calls spread by pairs over the group's devices (b200m_group_*_batch): Context's methods, with the
    # same arguments and results (each pair's output is what the Context method gives), over the group forms.  They
    # replace the sets uploaded before (every device then holds its own range's): match / knn raise until both sides are
    # uploaded again.
    knn_batch = Context.knn_batch
    match_batch = Context.match_batch
    match_wide_batch = Context.match_wide_batch
    match_wide_local_batch = Context.match_wide_local_batch
    _wide_batch = Context._wide_batch
    _params = staticmethod(Context._params)
    _pairs = staticmethod(Context._pairs)
    _scales = staticmethod(Context._scales)
    _WIDE_FIELDS = Context._WIDE_FIELDS
    _batch_sides = Context._batch_sides

    def _batch_call(self, name):
        self.n = [None, None]   # set before the call: a failed batch may have replaced the sets too
        return getattr(self._L, "b200m_group_" + name)

    def _batch_rows(self, counts):
        pass


_groups = threading.local()
_all_groups = []


def shared_group(devices):
    """One Group per host thread and device list, created on first use and kept (as the C++ shim's shared_group): creating a
    group starts a context and a thread per device and an NCCL communicator, which can cost more than a batch."""
    cache = _groups.__dict__.setdefault("by_devices", {})
    key = tuple(int(d) for d in devices)
    if key not in cache:
        cache[key] = Group(list(key))
        _all_groups.append(cache[key])
    return cache[key]


@atexit.register
def _close_groups():
    for g in _all_groups:
        g.close()


def batch_partition(cost, n_parts):
    """b200m_batch_partition: the contiguous split of pairs with these costs into n_parts ranges that the group batch calls
    use (pure host code).  -> int array first [n_parts + 1]; range i is [first[i], first[i + 1])."""
    c = np.ascontiguousarray(cost, np.float64)
    first = np.zeros(int(n_parts) + 1, np.int32)
    if load_library().b200m_batch_partition(c.ctypes.data, c.shape[0], int(n_parts), first.ctypes.data) != 0:
        raise B200MatchError("batch_partition: n_parts must be >= 1 and every cost finite and >= 0")
    return first


# ---- the reference's free functions ------------------------------------------------------
def _knn_once(query, train, dim, k, precision, device):
    with Context(device) as ctx:
        ctx.upload(0, query, dim)
        ctx.upload(1, train, dim)
        return ctx.knn(k, 0, precision=precision)


def match_bf(query_features, train_features, parameters, dim=None, device=0):
    """matchBF<FeatureT> (include/matching.h:594-634): per query the <= k nearest train rows, ascending L2
    distance.  Returns (match_indices [nq,k] -1 padded, distances [nq,k], count [nq]) -- the columns of the
    reference's std::vector<MultivaluedCorrespondence>.  Exact ties are ordered by lower train index (OpenCV's
    in-block rule; the reference's cross-block merge reverses them, see DESIGN.md)."""
    dim = dim or np.asarray(query_features).shape[1]
    return _knn_once(query_features, train_features, dim, parameters.randomness, parameters.precision, device)


def match_flann(query_features, train_features, parameters, dim=None, device=0):
    """matchFLANN<FeatureT> (include/matching.h:562-592): the same exact result set."""
    return match_bf(query_features, train_features, parameters, dim, device)


def match_local(query_features, train_features, parameters, dim=None, device=0, query_kps_xyz=None, train_kps_xyz=None,
                guess=None, match_search_radius=None):
    """matchLocal<FeatureT> (include/matching.h:637-678).  Without keypoints / radius: match_search_radius = inf, as
    the reference's test calls it (tests/flann_bf_matcher.h:66-72) == the plain exact kNN.  With them: only train rows
    whose keypoint lies within match_search_radius of the guess-transformed query keypoint are considered.  `guess`
    (4x4) is applied here in float32 (x' = R x + t); pass already transformed keypoints and guess=None to keep PCL's own
    transformPointCloudWithNormals arithmetic."""
    if query_kps_xyz is None or train_kps_xyz is None or match_search_radius is None or not np.isfinite(match_search_radius):
        return match_bf(query_features, train_features, parameters, dim, device)
    qx = np.ascontiguousarray(query_kps_xyz, np.float32)
    if guess is not None:
        g = np.asarray(guess, np.float32)
        moved = qx.copy()
        moved[:, :3] = qx[:, :3] @ g[:3, :3].T + g[:3, 3]
        qx = moved
    dim = dim or np.asarray(query_features).shape[1]
    with Context(device) as ctx:
        ctx.upload(0, query_features, dim)
        ctx.upload(1, train_features, dim)
        return ctx.knn_local(parameters.randomness, qx, train_kps_xyz, match_search_radius)


def match_multiscale(query_scales, train_scales, n_query_kps, train_kps_xyz, iss_radius, parameters, dim=None, device=0):
    """FeatureBasedMatcherImpl<FeatureT>::match_multiscale (include/matching.h:264-354) over precomputed per-scale
    descriptors: `query_scales` / `train_scales` are lists (one entry per common scale, ascending log2 radius) of
    (features [n_s, >= dim] float32, kps_indices [n_s] int32 or None) -- the reference's kps_features_multiscale[s] and
    kps_indices_multiscale[s].  Per scale an exact kNN (k = parameters.randomness), remapped to keypoint ids; then the
    spatial vote over the train keypoints' xyz keeps at most one match per query keypoint.
    Returns (match_index [n_query_kps] (-1: none), distance, count 0/1)."""
    if len(query_scales) != len(train_scales) or not query_scales:
        raise B200MatchError("match_multiscale: need the same, non-zero number of scales on both sides")
    xyz = np.ascontiguousarray(train_kps_xyz, np.float32)
    with Context(device) as ctx:
        ctx.multiscale_begin(n_query_kps, len(query_scales), parameters.randomness)
        for s, ((qf, qmap), (tf, tmap)) in enumerate(zip(query_scales, train_scales)):
            d = dim or np.asarray(qf).shape[1]
            ctx.upload(0, qf, d)
            ctx.upload(1, tf, d)
            ctx.multiscale_add(s, 0, qmap, tmap, xyz.shape[0], precision=parameters.precision)
        return ctx.multiscale_vote(xyz, iss_radius)


# ---- the reference's matcher classes --------------------------------------------------------
class FeatureBasedMatcher:
    """FeatureBasedMatcherImpl<FeatureT> (include/matching.h:96-161) at the descriptor seam: constructed over the two
    clouds' per-scale keypoint descriptors (the reference's `initialize` -- downsampling, normals, feature extraction --
    is out of scope).  match() = match_impl + finalize, and match_impl is composed as in the reference: match_multiscale
    (per-scale kNN with k = randomness, spatial vote -> at most one match per keypoint) in one or both directions, then
    the matcher's filter over the VOTED lists.

    src_features / tgt_features: one float32 array [n, >= dim] (a single scale) or a list of them (kps_features_multiscale,
    ascending scale); kps_indices_multiscale_src/tgt: the per-scale row -> keypoint id maps (None = identity);
    kps_xyz_src/tgt + iss_radius_src/tgt: keypoint coordinates and Storage::iss_radius, needed by the vote whenever a
    keypoint can have more than one candidate (randomness * scales > 1) and by the cluster filter;
    kps_indices_src/tgt: keypoint id -> cloud index (finalize)."""
    mode = None
    name = "FeatureBasedMatcher"

    def __init__(self, src_features, tgt_features, parameters, dim=None, thresholds_src=None, thresholds_tgt=None,
                 kps_indices_src=None, kps_indices_tgt=None, device=0, kps_xyz_src=None, kps_xyz_tgt=None,
                 iss_radius_src=None, iss_radius_tgt=None, kps_indices_multiscale_src=None, kps_indices_multiscale_tgt=None):
        self.parameters = parameters
        self.src = list(src_features) if isinstance(src_features, (list, tuple)) else [src_features]
        self.tgt = list(tgt_features) if isinstance(tgt_features, (list, tuple)) else [tgt_features]
        if len(self.src) != len(self.tgt) or not self.src:
            raise B200MatchError("the two clouds need the same, non-zero number of scales")
        self.dim = dim or np.asarray(self.src[0]).shape[1]
        self.thr_src, self.thr_tgt = thresholds_src, thresholds_tgt
        self.kps_src, self.kps_tgt = kps_indices_src, kps_indices_tgt
        self.xyz_src, self.xyz_tgt = kps_xyz_src, kps_xyz_tgt
        self.iss_src, self.iss_tgt = iss_radius_src, iss_radius_tgt
        self.maps_src = kps_indices_multiscale_src or [None] * len(self.src)
        self.maps_tgt = kps_indices_multiscale_tgt or [None] * len(self.tgt)
        self.device = device
        self.average_distance_ = FLT_MAX      # include/matching.h:41

    def get_average_distance(self):
        return self.average_distance_

    def get_class_name(self):
        return self.name

    def _k(self):
        return self.parameters.randomness

    def _uses_wide_seam(self):
        # _match_impl's route: without coordinates and radii only the k-list call of one candidate per keypoint is possible
        if self.xyz_src is not None and self.xyz_tgt is not None and self.iss_src is not None and self.iss_tgt is not None:
            return True
        if not self._vote_is_identity() or self.mode == MODE_CLUSTER:
            raise B200MatchError(
                "%s: randomness * scales > 1 (or the cluster filter) needs kps_xyz_src/tgt and iss_radius_src/tgt -- "
                "match_multiscale's spatial vote keeps one match per keypoint (reference include/matching.h:327-352)" % self.name)
        return False

    def _vote_is_identity(self):
        # one candidate per keypoint: the vote keeps it (its own term of the count is 1), include/matching.h:327-352
        return len(self.src) == 1 and self._k() == 1 and self.maps_src[0] is None and self.maps_tgt[0] is None

    def _match_impl(self, ctx):
        p = self.parameters
        if not self._uses_wide_seam():
            ctx.upload(0, self.src[0], self.dim)
            ctx.upload(1, self.tgt[0], self.dim)
            return ctx.match(1, self.mode, p.ratio_thr, p.distance_thr, self.thr_src, self.thr_tgt, p.precision, p.cand_cap)
        return ctx.match_wide(self._k(), self.mode, list(zip(self.src, self.maps_src)), list(zip(self.tgt, self.maps_tgt)),
                              self.xyz_src, self.xyz_tgt, self.iss_src, self.iss_tgt, self.dim, p.cluster_k, p.distance_thr,
                              self.thr_src, self.thr_tgt, p.precision, p.cand_cap)

    def _guess(self):
        """parameters.guess as float32 [4, 4], or None; refuses matchers that cannot take one (before any device is used)"""
        if self.parameters.guess is None:
            return None
        if self.mode not in (MODE_ONE_SIDED, MODE_MUTUAL, MODE_CLUSTER):
            raise B200MatchError("%s: a guess is not supported (the reference's RatioMatcher is a stub)" % self.name)
        if self.xyz_src is None or self.xyz_tgt is None or self.iss_src is None or self.iss_tgt is None:
            raise B200MatchError("%s: a guess needs kps_xyz_src/tgt and iss_radius_src/tgt -- matchLocal gates the candidates "
                                 "on the keypoint coordinates (reference include/matching.h:637-678)" % self.name)
        return guess_matrix(self.parameters.guess)

    def _wide_pair(self, g=None):
        """this matcher as one pair of Context.match_wide_batch, or with the guess g of match_wide_local_batch: the source
        keypoints moved by g, the target keypoints by its inverse"""
        pr = dict(src_scales=list(zip(self.src, self.maps_src)), tgt_scales=list(zip(self.tgt, self.maps_tgt)),
                  src_kps_xyz=self.xyz_src, tgt_kps_xyz=self.xyz_tgt, iss_radius_src=self.iss_src, iss_radius_tgt=self.iss_tgt)
        if g is not None:
            pr["src_kps_moved"] = transform_keypoints(self.xyz_src, g)
            pr["tgt_kps_moved"] = transform_keypoints(self.xyz_tgt, invert_guess(g))
        return pr

    def match(self):
        """match() (include/matching.h:148-161): match_impl + finalize (:356-362).  With parameters.guess set, match_impl's
        kNN is matchLocal's (one pair of Context.match_wide_local_batch)."""
        g = self._guess()
        with Context(self.device) as ctx:
            if g is None:
                corrs, avg = self._match_impl(ctx)
            else:
                p = self.parameters
                corrs, avg = ctx.match_wide_local_batch(self._k(), self.mode, [self._wide_pair(g)], p.match_search_radius, self.dim,
                                                        p.cluster_k, p.distance_thr, None if self.thr_src is None else [self.thr_src],
                                                        None if self.thr_tgt is None else [self.thr_tgt])[0]
        return self._finalize(corrs, avg)

    def _finalize(self, corrs, avg):
        corrs = corrs.copy()
        self.average_distance_ = avg
        if self.kps_src is not None:
            corrs["index_query"] = np.asarray(self.kps_src, np.int32)[corrs["index_query"]]
        if self.kps_tgt is not None:
            corrs["index_match"] = np.asarray(self.kps_tgt, np.int32)[corrs["index_match"]]
        return corrs


class OneSidedMatcher(FeatureBasedMatcher):
    """include/matching.h:385-416"""
    mode, name = MODE_ONE_SIDED, "OneSidedMatcher"


class LeftToRightMatcher(FeatureBasedMatcher):
    """include/matching.h:418-458"""
    mode, name = MODE_MUTUAL, "LeftToRightMatcher"


class ClusterMatcher(FeatureBasedMatcher):
    """ClusterMatcher (include/matching.h:480-551), the reference's default matching_id: always needs the keypoint
    coordinates of both sides (st_src_.kps / st_tgt_.kps); iss radii default to 1 when the vote is the identity."""
    mode, name = MODE_CLUSTER, "ClusterMatcher"

    def __init__(self, src_features, tgt_features, parameters, **kw):
        super().__init__(src_features, tgt_features, parameters, **kw)
        if self.xyz_src is None or self.xyz_tgt is None:
            raise B200MatchError("ClusterMatcher needs kps_xyz_src and kps_xyz_tgt (keypoint coordinates of both sides)")
        if self.iss_src is None or self.iss_tgt is None:
            if not self._vote_is_identity():
                raise B200MatchError("ClusterMatcher: randomness * scales > 1 needs iss_radius_src/tgt for the spatial vote")
            self.iss_src = self.iss_tgt = 1.0


class RatioMatcher(FeatureBasedMatcher):
    """A stub in the reference (include/matching.h:470-473: match_impl returns {}); semantics defined in DESIGN.md on the
    raw k-lists of a single scale (parity unpinned -- there is no reference behaviour)."""
    mode, name = MODE_RATIO, "RatioMatcher"

    def _k(self):
        return max(self.parameters.ratio_k, 2)

    def _match_impl(self, ctx):
        p = self.parameters
        if len(self.src) != 1:
            raise B200MatchError("RatioMatcher is defined on a single scale")
        ctx.upload(0, self.src[0], self.dim)
        ctx.upload(1, self.tgt[0], self.dim)
        return ctx.match(self._k(), self.mode, p.ratio_thr, p.distance_thr, self.thr_src, self.thr_tgt, p.precision, p.cand_cap)


def match_many(matchers, devices=None):
    """match() of many matchers at once (multi-view registration, one scan against many submaps, an evaluation table): one
    batch call instead of one call per matcher.  All matchers must be of one class, with equal AlignmentParameters (the guess
    aside: each matcher may have its own), dim and device.  Matchers with a guess go through Context.match_wide_local_batch;
    either every matcher has one or none has.  Without guesses, RatioMatchers and matchers whose vote is the identity and
    that have no keypoint coordinates go through Context.match_batch (as match() sends them to the k-list call), every other
    through Context.match_wide_batch.  Applies each matcher's finalize and sets its average distance; returns one
    correspondence array per matcher, each equal to what that matcher's match() returns.  devices: None (the matchers'
    device) or a list of device ids; with several, the batch is spread by pairs over them by this thread's shared_group of
    those devices (same results), with one, it runs on that device."""
    ms = list(matchers)
    if not ms:
        return []
    m0 = ms[0]
    unguessed = dataclasses.replace(m0.parameters, guess=None)
    for m in ms[1:]:
        if (type(m) is not type(m0) or dataclasses.replace(m.parameters, guess=None) != unguessed or m.dim != m0.dim
                or m.device != m0.device):
            raise B200MatchError("match_many: every matcher must be of one class, with equal AlignmentParameters, dim and device")
    if len({m.parameters.guess is None for m in ms}) > 1:
        raise B200MatchError("match_many: give every matcher a guess or none (the guessed and unguessed kNN are different calls)")
    p = m0.parameters

    def backend():
        if devices and len(devices) > 1:
            return contextlib.nullcontext(shared_group(devices))
        return Context(devices[0] if devices else m0.device)

    if p.guess is not None:
        guesses = [m._guess() for m in ms]
        ts = None if all(m.thr_src is None and m.thr_tgt is None for m in ms) else [
            np.full(len(m.xyz_src), np.inf, np.float32) if m.thr_src is None else m.thr_src for m in ms]
        tt = None if ts is None else [np.full(len(m.xyz_tgt), np.inf, np.float32) if m.thr_tgt is None else m.thr_tgt for m in ms]
        with backend() as ctx:
            got = ctx.match_wide_local_batch(m0._k(), m0.mode, [m._wide_pair(g) for m, g in zip(ms, guesses)],
                                             p.match_search_radius, m0.dim, p.cluster_k, p.distance_thr, ts, tt)
        return [m._finalize(*r) for m, r in zip(ms, got)]
    narrow, wide = [], []
    for i, m in enumerate(ms):
        if isinstance(m, RatioMatcher):
            if len(m.src) != 1:
                raise B200MatchError("RatioMatcher is defined on a single scale")
            narrow.append(i)
        else:
            (wide if m._uses_wide_seam() else narrow).append(i)

    def thresholds(group):
        # a matcher without thresholds gets +inf ones: min(max(inf, .), distance_thr) is distance_thr, as with none
        if all(ms[i].thr_src is None and ms[i].thr_tgt is None for i in group):
            return None, None
        ts, tt = [], []
        for i in group:
            m = ms[i]
            if (m.thr_src is None) != (m.thr_tgt is None):
                raise B200MatchError("%s: give both threshold arrays or neither" % m.name)
            n_s, n_t = (len(m.src[0]), len(m.tgt[0])) if i in narrow else (len(m.xyz_src), len(m.xyz_tgt))
            ts.append(np.full(n_s, np.inf, np.float32) if m.thr_src is None else m.thr_src)
            tt.append(np.full(n_t, np.inf, np.float32) if m.thr_tgt is None else m.thr_tgt)
        return ts, tt

    results = [None] * len(ms)
    with backend() as ctx:
        if narrow:
            ts, tt = thresholds(narrow)
            k = m0._k() if isinstance(m0, RatioMatcher) else 1
            got = ctx.match_batch(k, m0.mode, [(ms[i].src[0], ms[i].tgt[0]) for i in narrow], m0.dim, p.ratio_thr, p.distance_thr,
                                  ts, tt, p.precision, p.cand_cap)
            for i, r in zip(narrow, got):
                results[i] = r
        if wide:
            ts, tt = thresholds(wide)
            got = ctx.match_wide_batch(m0._k(), m0.mode, [ms[i]._wide_pair() for i in wide], m0.dim, p.cluster_k, p.distance_thr, ts, tt, p.precision,
                                       p.cand_cap)
            for i, r in zip(wide, got):
                results[i] = r
    return [m._finalize(*r) for m, r in zip(ms, results)]


def get_feature_based_matcher_from_parameters(src_features, tgt_features, parameters, **kw):
    """getFeatureBasedMatcherFromParameters (src/matching.cpp:21-76) for the matchers on the hot path."""
    m = parameters.matching_id
    if m == MATCHING_ONE_SIDED:
        return OneSidedMatcher(src_features, tgt_features, parameters, **kw)
    if m == MATCHING_LEFT_TO_RIGHT:
        return LeftToRightMatcher(src_features, tgt_features, parameters, **kw)
    if m == MATCHING_RATIO:
        return RatioMatcher(src_features, tgt_features, parameters, **kw)
    if m == MATCHING_CLUSTER:
        return ClusterMatcher(src_features, tgt_features, parameters, **kw)
    raise B200MatchError("Matching method %s isn't supported by the B200 matcher" % m)
