"""ctypes binding of libgsc_cuda.so (include/gsc_cuda.h).

This is the Python face of the C ABI; there is NO CPU fallback here or in the
library: if the shared object is missing, or no sm_100 device is usable, every
call raises.  numpy arrays in, numpy arrays out.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# GSC_CUDA_SO: load another build of the same library (tools/spill_probe.py uses register-capped debug builds)
SO_PATH = os.environ.get("GSC_CUDA_SO") or os.path.join(_HERE, "libgsc_cuda.so")

#: every symbol include/gsc_cuda.h declares (checked by the CPU test-suite)
EXPORTS = [
    "yakmo_create", "yakmo_destroy", "yakmo_load_train_data", "yakmo_train_on_data", "yakmo_get_centroids",
    "ann_kdtree_create", "ann_kdtree_destroy", "ann_kdtree_search", "ann_kdtree_pri_search",
    "ann_kdtree_search_multi", "ann_kdtree_pri_search_multi",
    "gsc_last_error", "gsc_device_count", "gsc_create", "gsc_destroy", "gsc_ctx_device", "gsc_ctx_stream",
    "gsc_synchronize", "gsc_get_stats", "gsc_stage_busy_ms", "gsc_reset_stats",
    "gsc_find_attenuation_divider", "gsc_make_chunks", "gsc_yakmo", "gsc_knn_scan_reduce", "gsc_knn_scan_reduce_kdtree", "gsc_lloyd",
    "gsc_assign", "gsc_split_begin", "gsc_split_step", "gsc_split_update", "gsc_split_end",
    "gsc_split_unique_id", "gsc_split_comm_init", "gsc_split_comm_destroy", "gsc_split_seed", "gsc_split_lloyd", "gsc_build_dictionary", "gsc_knnfit", "gsc_knnfit_kdtree", "gsc_finalize_dictionary",
    "gsc_default_params", "gsc_dict_capacity", "gsc_encode_frames", "gsc_encode_frames_dev",
    "gsc_fetch_results", "gsc_fetch_stream", "gsc_fetch_quality", "gsc_fp32_peak_probe", "gsc_log_array", "gsc_plan_frames", "gsc_plan_frames_dev", "gsc_ctx_set_debug", "gsc_selftest_divider_division", "gsc_debug_online_counters", "gsc_debug_seed_counters",
]


class GscError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [("chunk_size", C.c_int32), ("chunk_bit_depth", C.c_int32), ("chunks_per_frame", C.c_int32),
                ("precision", C.c_int32), ("max_passes", C.c_int32), ("kmeans_mode", C.c_int32),
                ("lloyd_iters", C.c_int32), ("reserved", C.c_int32)]


class FrameDesc(C.Structure):
    _fields_ = [("pcm", C.c_void_p), ("stride", C.c_int64), ("channels", C.c_int32), ("samples", C.c_int32)]


class FrameResultC(C.Structure):
    _fields_ = [("dict", C.c_void_p), ("datten", C.c_void_p), ("index", C.c_void_p), ("attr", C.c_void_p),
                ("N", C.c_int32), ("R", C.c_int32), ("divider", C.c_int32), ("passes", C.c_int32),
                ("err", C.c_double), ("overfull", C.c_int32), ("reserved", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("last_stage_ms", C.c_double * 8)]


STAGE_NAMES = ["divider", "chunks", "seed", "kmeans", "dictionary", "knnfit", "finalize", "total"]


@dataclass
class FrameResult:
    N: int
    R: int
    divider: int
    passes: int
    err: float
    dict: np.ndarray      # int16 [R][cs]
    datten: np.ndarray    # uint8 [R]
    index: np.ndarray     # int32 [N]
    attr: np.ndarray      # uint8 [N]  bit1 Negative, bit0 Reversed
    overfull: int


_lib = None


def load_library() -> C.CDLL:
    """Load libgsc_cuda.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise GscError(f"{SO_PATH} is missing: build it with `python -m soundchunks_b200.build` "
                       "(there is no CPU fallback)")
    L = C.CDLL(SO_PATH)
    L.gsc_last_error.restype = C.c_char_p
    L.gsc_create.restype = C.c_void_p
    L.gsc_create.argtypes = [C.c_int]
    L.gsc_destroy.argtypes = [C.c_void_p]
    L.gsc_ctx_stream.restype = C.c_void_p
    L.gsc_ctx_stream.argtypes = [C.c_void_p]
    L.gsc_ctx_device.argtypes = [C.c_void_p]
    L.gsc_synchronize.argtypes = [C.c_void_p]
    L.gsc_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    L.gsc_reset_stats.argtypes = [C.c_void_p]
    L.yakmo_create.restype = C.c_void_p
    L.yakmo_create.argtypes = [C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    L.yakmo_destroy.argtypes = [C.c_void_p]
    L.yakmo_load_train_data.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    L.yakmo_train_on_data.argtypes = [C.c_void_p, C.c_void_p]
    L.yakmo_get_centroids.argtypes = [C.c_void_p, C.c_void_p]
    L.ann_kdtree_create.restype = C.c_void_p
    L.ann_kdtree_create.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    L.ann_kdtree_destroy.argtypes = [C.c_void_p]
    for n in ("ann_kdtree_search", "ann_kdtree_pri_search"):
        getattr(L, n).restype = C.c_int32
        getattr(L, n).argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
    for n in ("ann_kdtree_search_multi", "ann_kdtree_pri_search_multi"):
        getattr(L, n).restype = None
        getattr(L, n).argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_float]
    _lib = L
    return L


def _vp(a: Optional[np.ndarray]):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _pcm(pcm) -> np.ndarray:
    pcm = np.ascontiguousarray(pcm, dtype=np.int16)
    if pcm.ndim == 1:
        pcm = pcm[None, :]
    return pcm


def device_count() -> int:
    return int(load_library().gsc_device_count())


def default_params(**kw) -> Params:
    p = Params()
    load_library().gsc_default_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


class Context:
    """One device + stream + scratch (gsc_ctx)."""

    def __init__(self, device: int = -1):
        self.L = load_library()
        self.h = self.L.gsc_create(device)
        if not self.h:
            raise GscError(self.L.gsc_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.gsc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc: int):
        if rc != 0:
            raise GscError(f"libgsc_cuda error {rc}: {self.L.gsc_last_error().decode()}")

    @property
    def device(self) -> int:
        return int(self.L.gsc_ctx_device(self.h))

    @property
    def stream(self) -> int:
        return int(self.L.gsc_ctx_stream(self.h) or 0)

    def synchronize(self):
        self._ck(self.L.gsc_synchronize(self.h))

    def stats(self) -> dict:
        s = Stats()
        self._ck(self.L.gsc_get_stats(self.h, C.byref(s)))
        return dict(kernel_launches=int(s.kernel_launches), h2d_bytes=int(s.h2d_bytes),
                    d2h_bytes=int(s.d2h_bytes),
                    stage_ms={n: float(s.last_stage_ms[i]) for i, n in enumerate(STAGE_NAMES)})

    def stage_busy_ms(self, stage: str) -> float:
        """Wall-clock ms during which `stage` of the last batch ran on at least one of the two internal streams."""
        v = C.c_double(0)
        self._ck(self.L.gsc_stage_busy_ms(C.c_void_p(self.h), STAGE_NAMES.index(stage), C.byref(v)))
        return v.value

    def reset_stats(self):
        self._ck(self.L.gsc_reset_stats(self.h))

    def online_counters(self, n_frames: int) -> np.ndarray:
        out = np.zeros((n_frames, 16), np.uint64)
        self._ck(self.L.gsc_debug_online_counters(C.c_void_p(self.h), _vp(out), n_frames))
        return out

    DBG_ONLINE_EXACT, DBG_SEED_FULLSCAN, DBG_SEED_SERIAL, DBG_KNNFIT_DENSE, DBG_LLOYD_OWNER, DBG_ONLINE_BATCHED, DBG_LABEL_SCAN, DBG_DIVIDER_V1 = 1, 2, 4, 8, 16, 32, 64, 128
    DBG_KDTREE_SERIAL = 256

    def set_debug(self, flags: int):
        """Cross-check paths (include/gsc_cuda.h GSC_DBG_*); 0 = the product path."""
        self._ck(self.L.gsc_ctx_set_debug(C.c_void_p(self.h), C.c_uint(flags)))

    def selftest_divider_division(self, bits: int) -> int:
        v = C.c_uint64(0)
        self._ck(self.L.gsc_selftest_divider_division(C.c_void_p(self.h), bits, C.byref(v)))
        return int(v.value)

    def seed_counters(self, n_frames: int) -> np.ndarray:
        out = np.zeros((n_frames, 8), np.uint64)
        self._ck(self.L.gsc_debug_seed_counters(C.c_void_p(self.h), _vp(out), n_frames))
        return out

    def plan_frames(self, pcm, sample_rate, frame_length_ms=4000.0, vfr=1.0, block=4, max_frames=None, return_stats=False):
        """enc:1374-1425 on the device: pcm planar int16 [C][S] (S padded to the block size) -> frame starts."""
        pcm = _pcm(pcm)
        Cn, S = pcm.shape
        if max_frames is None:
            max_frames = 4 * int(np.ceil(S / (sample_rate * frame_length_ms / 1000.0))) + 16
        starts = np.zeros(max_frames, np.int64)
        n = C.c_int(0)
        st = (C.c_uint64 * 4)()
        self._ck(self.L.gsc_plan_frames(C.c_void_p(self.h), _vp(pcm), C.c_int64(S), Cn, C.c_int64(S), sample_rate,
                                        C.c_double(frame_length_ms), C.c_double(vfr), block, _vp(starts), max_frames, C.byref(n), st))
        out = starts[:n.value].copy()
        return (out, dict(exact_windows_pass1=int(st[0]), exact_windows_pass2=int(st[1]), boundary_iterations=int(st[2]),
                          windows_pass1=int(st[3]))) if return_stats else out

    def log_array(self, x) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros_like(x)
        self._ck(self.L.gsc_log_array(C.c_void_p(self.h), _vp(x), C.c_int64(x.size), _vp(y)))
        return y

    def fp32_peak_tflops(self) -> float:
        v = C.c_double(0)
        self._ck(self.L.gsc_fp32_peak_probe(C.c_void_p(self.h), C.byref(v)))
        return v.value

    # ---- per-frame stages -------------------------------------------------
    def find_attenuation_divider(self, pcm, cs=4, bits=12, return_v=False):
        pcm = _pcm(pcm)
        Cn, S = pcm.shape
        d = C.c_int(0)
        v = np.zeros(64, np.float64)
        self._ck(self.L.gsc_find_attenuation_divider(C.c_void_p(self.h), _vp(pcm), C.c_int64(S), Cn, S, cs, bits,
                                                     C.byref(d), _vp(v)))
        return (d.value, v) if return_v else d.value

    def make_chunks(self, pcm, cs=4, bits=12, divider=6):
        """-> attr u8[N], atten u8[N], feat f32[N][2cs], dst i16[N][cs]"""
        pcm = _pcm(pcm)
        Cn, S = pcm.shape
        N = ((S - 1) // cs + 1) * Cn
        attr = np.zeros(N, np.uint8)
        atten = np.zeros(N, np.uint8)
        feat = np.zeros((N, 2 * cs), np.float32)
        dst = np.zeros((N, cs), np.int16)
        self._ck(self.L.gsc_make_chunks(C.c_void_p(self.h), _vp(pcm), C.c_int64(S), Cn, S, cs, bits, divider,
                                        _vp(attr), _vp(atten), _vp(feat), _vp(dst)))
        return attr, atten, feat, dst

    def yakmo(self, X, K, init_type=1, max_iter=0):
        X = np.ascontiguousarray(X, dtype=np.float32)
        N, D = X.shape
        cen = np.zeros((K, D), np.float32)
        labels = np.zeros(N, np.int32)
        seeds = np.zeros(K, np.int32)
        self._ck(self.L.gsc_yakmo(C.c_void_p(self.h), _vp(X), N, D, K, init_type, max_iter, _vp(cen), _vp(labels),
                                  _vp(seeds)))
        return cen, labels, seeds

    def knn_scan_reduce(self, X, centroids, precision=3, max_passes=100):
        X = np.ascontiguousarray(X, dtype=np.float32)
        cen = np.array(centroids, dtype=np.float32, order="C", copy=True)
        N, D = X.shape
        labels = np.zeros(N, np.int32)
        passes = C.c_int(0)
        err = C.c_double(0)
        self._ck(self.L.gsc_knn_scan_reduce(C.c_void_p(self.h), _vp(X), N, D, _vp(cen), cen.shape[0], precision,
                                            max_passes, _vp(labels), C.byref(passes), C.byref(err)))
        return cen, labels, passes.value, err.value

    def knn_scan_reduce_kdtree(self, X, centroids, precision=3, max_passes=100):
        """kmeans_mode 3: KNNScanReduce through the reference's ANN kd-tree -> (centroids, labels, passes, err)"""
        X = np.ascontiguousarray(X, dtype=np.float32)
        cen = np.array(centroids, dtype=np.float32, order="C", copy=True)
        N, D = X.shape
        labels = np.zeros(N, np.int32)
        passes = C.c_int(0)
        err = C.c_double(0)
        self._ck(self.L.gsc_knn_scan_reduce_kdtree(C.c_void_p(self.h), _vp(X), N, D, _vp(cen), cen.shape[0], precision,
                                                   max_passes, _vp(labels), C.byref(passes), C.byref(err)))
        return cen, labels, passes.value, err.value

    def lloyd(self, X, centroids, iters):
        X = np.ascontiguousarray(X, dtype=np.float32)
        cen = np.array(centroids, dtype=np.float32, order="C", copy=True)
        N, D = X.shape
        labels = np.zeros(N, np.int32)
        self._ck(self.L.gsc_lloyd(C.c_void_p(self.h), _vp(X), N, D, _vp(cen), cen.shape[0], iters, _vp(labels)))
        return cen, labels

    # ---- oversized frame split over GPUs (one Context per rank) ------------
    def split_begin(self, X, centroids):
        X = np.ascontiguousarray(X, dtype=np.float32)
        cen = np.ascontiguousarray(centroids, dtype=np.float32)
        self._split = (X.shape[0], X.shape[1], cen.shape[0])
        self._ck(self.L.gsc_split_begin(C.c_void_p(self.h), _vp(X), X.shape[0], X.shape[1], _vp(cen), cen.shape[0]))

    def split_step(self, acc_dev_ptr: int):
        self._ck(self.L.gsc_split_step(C.c_void_p(self.h), C.c_void_p(acc_dev_ptr)))

    def split_update(self, acc_dev_ptr: int):
        self._ck(self.L.gsc_split_update(C.c_void_p(self.h), C.c_void_p(acc_dev_ptr)))

    def split_end(self):
        N, D, K = self._split
        cen = np.zeros((K, D), np.float32)
        labels = np.zeros(N, np.int32)
        self._ck(self.L.gsc_split_end(C.c_void_p(self.h), _vp(cen), _vp(labels)))
        return cen, labels

    # ---- the same with NCCL inside the library (gsc_split_lloyd) ------------
    @staticmethod
    def split_unique_id() -> bytes:
        L = load_library()
        buf = C.create_string_buffer(128)
        if L.gsc_split_unique_id(buf) != 0:
            raise GscError(L.gsc_last_error().decode())
        return buf.raw

    def split_comm_init(self, nranks: int, rank: int, uid: bytes):
        self._ck(self.L.gsc_split_comm_init(C.c_void_p(self.h), nranks, rank, C.c_char_p(uid)))

    def split_comm_destroy(self):
        self._ck(self.L.gsc_split_comm_destroy(C.c_void_p(self.h)))

    def split_seed(self, X_shard, K):
        X = np.ascontiguousarray(X_shard, dtype=np.float32)
        cen = np.zeros((K, X.shape[1]), np.float32)
        self._ck(self.L.gsc_split_seed(C.c_void_p(self.h), _vp(X), X.shape[0], X.shape[1], K, _vp(cen)))
        return cen

    def split_lloyd(self, X_shard, centroids, iters):
        """-> (centroids, labels of the shard, dict(ms_loop, ms_allreduce, ms_first_iter))"""
        X = np.ascontiguousarray(X_shard, dtype=np.float32)
        cen = np.array(centroids, dtype=np.float32, order="C", copy=True)
        labels = np.zeros(X.shape[0], np.int32)
        ms = (C.c_double * 3)()
        self._ck(self.L.gsc_split_lloyd(C.c_void_p(self.h), _vp(X), X.shape[0], X.shape[1], _vp(cen), cen.shape[0], iters,
                                        _vp(labels), ms))
        return cen, labels, dict(ms_loop=ms[0], ms_allreduce=ms[1], ms_first_iter=ms[2])

    def assign(self, X, centroids):
        X = np.ascontiguousarray(X, dtype=np.float32)
        cen = np.ascontiguousarray(centroids, dtype=np.float32)
        N, D = X.shape
        labels = np.zeros(N, np.int32)
        dist = np.zeros(N, np.float32)
        self._ck(self.L.gsc_assign(C.c_void_p(self.h), _vp(X), N, D, _vp(cen), cen.shape[0], _vp(labels), _vp(dist)))
        return labels, dist

    def build_dictionary(self, labels, pcm, attr, K, cs=4, bits=12, divider=6):
        pcm = _pcm(pcm)
        Cn, S = pcm.shape
        labels = np.ascontiguousarray(labels, dtype=np.int32)
        attr = np.ascontiguousarray(attr, dtype=np.uint8)
        N = len(labels)
        out = dict(means=np.zeros((K, cs), np.float32), order=np.zeros(K, np.int32), counts=np.zeros(K, np.int32),
                   dict=np.zeros((K, cs), np.int16), datten=np.zeros(K, np.uint8), dattr=np.zeros(K, np.uint8),
                   entry=np.zeros(N, np.int32))
        self._ck(self.L.gsc_build_dictionary(C.c_void_p(self.h), _vp(labels), _vp(pcm), C.c_int64(S), Cn, S, _vp(attr),
                                             cs, K, bits, divider, _vp(out["means"]), _vp(out["order"]),
                                             _vp(out["counts"]), _vp(out["dict"]), _vp(out["datten"]),
                                             _vp(out["dattr"]), _vp(out["entry"])))
        return out

    def knnfit(self, dic, datten, pcm, cs=4, bits=12, divider=6):
        pcm = _pcm(pcm)
        Cn, S = pcm.shape
        dic = np.ascontiguousarray(dic, dtype=np.int16)
        datten = np.ascontiguousarray(datten, dtype=np.uint8)
        R = dic.shape[0]
        N = ((S - 1) // cs + 1) * Cn
        out = dict(best=np.zeros(N, np.int32), use=np.zeros(R, np.int32), band=np.zeros(N, np.int32))
        self._ck(self.L.gsc_knnfit(C.c_void_p(self.h), _vp(dic), _vp(datten), R, cs, bits, divider, _vp(pcm),
                                   C.c_int64(S), Cn, S, _vp(out["best"]), _vp(out["use"]), _vp(out["band"])))
        return out

    def knnfit_kdtree(self, dic, datten, pcm, cs=4, bits=12, divider=6):
        """kmeans_mode 3: KNNFit through the reference's ANN kd-tree (64 nearest rows) -> dict(best, use)"""
        pcm = _pcm(pcm)
        Cn, S = pcm.shape
        dic = np.ascontiguousarray(dic, dtype=np.int16)
        datten = np.ascontiguousarray(datten, dtype=np.uint8)
        R = dic.shape[0]
        N = ((S - 1) // cs + 1) * Cn
        out = dict(best=np.zeros(N, np.int32), use=np.zeros(R, np.int32))
        self._ck(self.L.gsc_knnfit_kdtree(C.c_void_p(self.h), _vp(dic), _vp(datten), R, cs, bits, divider, _vp(pcm),
                                          C.c_int64(S), Cn, S, _vp(out["best"]), _vp(out["use"])))
        return out

    def finalize_dictionary(self, use):
        use = np.ascontiguousarray(use, dtype=np.int32)
        R = len(use)
        remap = np.zeros(R, np.int32)
        order = np.zeros(R, np.int32)
        n = C.c_int(0)
        self._ck(self.L.gsc_finalize_dictionary(C.c_void_p(self.h), _vp(use), R, _vp(remap), _vp(order), C.byref(n)))
        return n.value, remap, order[:n.value]

    # ---- whole frames -------------------------------------------------------
    def encode_frames(self, frames: Sequence[np.ndarray], params: Optional[Params] = None, **kw) -> List[FrameResult]:
        """frames: list of planar int16 [C][S] arrays (host). One gsc_encode_frames call."""
        p = params if params is not None else default_params(**kw)
        fr = [_pcm(f) for f in frames]
        n = len(fr)
        desc = (FrameDesc * n)()
        res = (FrameResultC * n)()
        cap = int(self.L.gsc_dict_capacity(C.byref(p), 0, 0))
        cs = p.chunk_size
        bufs = []
        for i, f in enumerate(fr):
            Cn, S = f.shape
            N = ((S - 1) // cs + 1) * Cn
            desc[i] = FrameDesc(f.ctypes.data, S, Cn, S)
            d = np.zeros((max(cap, 1), cs), np.int16)
            a = np.zeros(max(cap, 1), np.uint8)
            ix = np.zeros(N, np.int32)
            at = np.zeros(N, np.uint8)
            bufs.append((d, a, ix, at))
            res[i].dict, res[i].datten, res[i].index, res[i].attr = d.ctypes.data, a.ctypes.data, ix.ctypes.data, at.ctypes.data
        self._ck(self.L.gsc_encode_frames(C.c_void_p(self.h), desc, n, C.byref(p), res))
        out = []
        for i in range(n):
            d, a, ix, at = bufs[i]
            R = res[i].R
            out.append(FrameResult(N=res[i].N, R=R, divider=res[i].divider, passes=res[i].passes, err=res[i].err,
                                   dict=d[:R].copy(), datten=a[:R].copy(), index=ix, attr=at,
                                   overfull=res[i].overfull))
        return out

    def fetch_stream(self, n_frames: int, sample_rate: int):
        """.gsc bytes of the last batch, packed on the device -> (bytearray, per-frame sizes)."""
        sizes = np.zeros(n_frames, np.int64)
        total = C.c_int64(0)
        # sizing call: packs on the device and brings back 8 bytes per frame; the second call copies the bytes (once)
        self._ck(self.L.gsc_fetch_stream(C.c_void_p(self.h), n_frames, sample_rate, None, C.c_int64(0), _vp(sizes), C.byref(total)))
        out = bytearray(max(total.value, 1))        # the library writes straight into it: no second host copy
        buf = (C.c_char * len(out)).from_buffer(out)
        self._ck(self.L.gsc_fetch_stream(C.c_void_p(self.h), n_frames, sample_rate, C.cast(buf, C.c_void_p), C.c_int64(total.value),
                                         _vp(sizes), C.byref(total)))
        del buf
        if total.value != len(out):
            del out[total.value:]
        return out, sizes

    def fetch_quality(self, n_frames: int):
        """-> (sum of squared int16 errors per frame, samples per frame); PsyADelta = sqrt(sum / sum)."""
        e2 = np.zeros(n_frames, np.uint64)
        ns = np.zeros(n_frames, np.int64)
        self._ck(self.L.gsc_fetch_quality(C.c_void_p(self.h), n_frames, _vp(e2), _vp(ns)))
        return e2, ns

    def encode_to_stream(self, frames: Sequence[np.ndarray], sample_rate: int, params: Optional[Params] = None, **kw):
        """Host PCM in, .gsc bytes out (gsc_encode_frames without per-frame results + gsc_fetch_stream): what
        an encoder front-end needs.  -> (bytes, per-frame sizes)"""
        p = params if params is not None else default_params(**kw)
        fr = [_pcm(f) for f in frames]
        n = len(fr)
        desc = (FrameDesc * n)()
        for i, f in enumerate(fr):
            desc[i] = FrameDesc(f.ctypes.data, f.shape[1], f.shape[0], f.shape[1])
        self._ck(self.L.gsc_encode_frames(C.c_void_p(self.h), desc, n, C.byref(p), None))
        return self.fetch_stream(n, sample_rate)

    def encode_frames_dev(self, dev_ptr: int, layout: Sequence[tuple], params: Params):
        """Device-resident PCM: layout = [(offset_samples, stride, channels, samples), ...] into the
        int16 buffer at dev_ptr.  Results stay on the device (fetch_results)."""
        n = len(layout)
        desc = (FrameDesc * n)()
        for i, (off, stride, Cn, S) in enumerate(layout):
            desc[i] = FrameDesc(dev_ptr + 2 * off, stride, Cn, S)
        self._ck(self.L.gsc_encode_frames_dev(C.c_void_p(self.h), desc, n, C.byref(params)))

    def fetch_results(self, layout: Sequence[tuple], params: Params) -> List[FrameResult]:
        n = len(layout)
        res = (FrameResultC * n)()
        cap = int(self.L.gsc_dict_capacity(C.byref(params), 0, 0))
        cs = params.chunk_size
        bufs = []
        for i, (off, stride, Cn, S) in enumerate(layout):
            N = ((S - 1) // cs + 1) * Cn
            d = np.zeros((max(cap, 1), cs), np.int16)
            a = np.zeros(max(cap, 1), np.uint8)
            ix = np.zeros(N, np.int32)
            at = np.zeros(N, np.uint8)
            bufs.append((d, a, ix, at))
            res[i].dict, res[i].datten, res[i].index, res[i].attr = d.ctypes.data, a.ctypes.data, ix.ctypes.data, at.ctypes.data
        self._ck(self.L.gsc_fetch_results(C.c_void_p(self.h), n, res))
        out = []
        for i in range(n):
            d, a, ix, at = bufs[i]
            R = res[i].R
            out.append(FrameResult(N=res[i].N, R=R, divider=res[i].divider, passes=res[i].passes, err=res[i].err,
                                   dict=d[:R].copy(), datten=a[:R].copy(), index=ix, attr=at,
                                   overfull=res[i].overfull))
        return out


# ---- legacy ABI helpers (what extern.pas binds) ------------------------------
def _row_ptrs(a: np.ndarray):
    rows = (C.c_void_p * a.shape[0])()
    base = a.ctypes.data
    stride = a.strides[0]
    for i in range(a.shape[0]):
        rows[i] = base + i * stride
    return rows


def legacy_yakmo(X: np.ndarray, k: int, max_iter: int = 0, init_type: int = 1):
    """yakmo_create .. yakmo_destroy exactly as enc:824-828 drives them."""
    L = load_library()
    X = np.ascontiguousarray(X, dtype=np.float32)
    N, D = X.shape
    h = L.yakmo_create(k, 1, max_iter, init_type, 0, 0, 0)
    if not h:
        raise GscError(L.gsc_last_error().decode())
    try:
        L.yakmo_load_train_data(h, N, D, _row_ptrs(X))
        labels = np.zeros(N, np.int32)
        L.yakmo_train_on_data(h, _vp(labels))
        cen = np.zeros((k, D), np.float32)
        L.yakmo_get_centroids(h, _row_ptrs(cen))
    finally:
        L.yakmo_destroy(h)
    return cen, labels


class LegacyAnn:
    """ann_kdtree_* as ext:118-123 binds them."""

    def __init__(self, pts: np.ndarray, copy: bool = True):
        """copy=False: the handle aliases the rows of `pts` itself (a C-contiguous float32 array the caller goes on
        mutating, as enc:736-740 does); the row-pointer table is kept alive with the handle."""
        self.L = load_library()
        self.pts = np.ascontiguousarray(pts, dtype=np.float32) if copy else pts
        assert self.pts.dtype == np.float32 and self.pts.flags.c_contiguous
        n, dd = self.pts.shape
        self._rows = _row_ptrs(self.pts)
        self.h = self.L.ann_kdtree_create(self._rows, n, dd, 1, 0)
        if not self.h:
            raise GscError(self.L.gsc_last_error().decode())

    def search(self, q):
        q = np.ascontiguousarray(q, dtype=np.float32)
        err = C.c_float(0)
        idx = self.L.ann_kdtree_search(self.h, _vp(q), 0.0, C.byref(err))
        return int(idx), float(err.value)

    def pri_search_multi(self, q, cnt):
        q = np.ascontiguousarray(q, dtype=np.float32)
        idxs = np.zeros(cnt, np.int32)
        errs = np.zeros(cnt, np.float32)
        self.L.ann_kdtree_pri_search_multi(self.h, _vp(idxs), _vp(errs), cnt, _vp(q), 0.0)
        return idxs, errs

    def close(self):
        if self.h:
            self.L.ann_kdtree_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
