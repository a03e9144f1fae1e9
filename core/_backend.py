"""ctypes binding of libtnn_b200.so (include/tnn_b200.h) and the device array type.

This module is the only place the host side touches the GPU.  There is no CPU fallback: if the
shared library is missing, cannot be loaded, or no sm_100 device is present, the first operation
raises.  The reference's numpy calls in core/ops.py map onto the functions here one to one
(citations in include/tnn_b200.h).
"""
import ctypes
import gc
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get(
    "TNN_B200_LIB", os.path.join(_ROOT, "tinynn-autograd_b200", "libtnn_b200.so"))

F32 = np.dtype(np.float32)
F64 = np.dtype(np.float64)
_DT_CODE = {F32: 0, F64: 1}
MAX_DIMS = 8

# op codes (include/tnn_b200.h)
ADD, SUB, MUL, DIV, POW, MAXIMUM, MINIMUM, GE, GT, LE, LT, EQ = range(12)
MUL_GE, MUL_GT, MUL_LE, MUL_LT, MUL_EQ, DIV_BWD_B, POW_BWD_A, POW_BWD_B = range(20, 28)
NEG, EXP, LOG, COPY, CLIP, SCALE, CLIP_BWD, RECIP_MUL = range(40, 48)
LEAKY_RELU, ELU, GELU, GELU_TANH, SOFTPLUS, SILU = range(48, 54)
LEAKY_RELU_BWD, ELU_BWD, GELU_BWD, GELU_TANH_BWD, SOFTPLUS_BWD, SILU_BWD = range(60, 66)
RED_SUM, RED_MAX, RED_MIN = 0, 1, 2
OPT_SGD, OPT_ADAM, OPT_RMSPROP, OPT_MOMENTUM, OPT_ADAGRAD, OPT_ADADELTA, OPT_ADAMW, OPT_RADAM, OPT_ADAMAX = range(9)

_c_i64 = ctypes.c_int64
_c_i32 = ctypes.c_int32
_c_int = ctypes.c_int
_c_vp = ctypes.c_void_p
_c_dbl = ctypes.c_double
_c_sz = ctypes.c_size_t

_lib = None
_inited = False


class BackendError(RuntimeError):
    pass


_SIGNATURES = {
    "tnn_init": [_c_int],
    "tnn_shutdown": [],
    "tnn_sync": [],
    "tnn_device_info": [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp],
    "tnn_device_count": [_c_vp],
    "tnn_alloc": [_c_sz, _c_vp],
    "tnn_free": [_c_vp],
    "tnn_pool_stats": [_c_vp, _c_vp, _c_vp],
    "tnn_pool_trim": [],
    "tnn_h2d": [_c_vp, _c_vp, _c_sz],
    "tnn_d2h": [_c_vp, _c_vp, _c_sz],
    "tnn_d2d": [_c_vp, _c_vp, _c_sz],
    "tnn_memset": [_c_vp, _c_int, _c_sz],
    "tnn_host_alloc": [_c_sz, _c_vp],
    "tnn_host_free": [_c_vp],
    "tnn_host_register": [_c_vp, _c_sz],
    "tnn_host_unregister": [_c_vp],
    "tnn_h2d_async_copy_stream": [_c_vp, _c_vp, _c_sz],
    "tnn_copy_stream_sync": [],
    "tnn_copy_wait_compute": [],
    "tnn_compute_wait_copy": [],
    "tnn_event_create": [_c_vp],
    "tnn_event_destroy": [_c_vp],
    "tnn_event_record": [_c_vp],
    "tnn_event_elapsed_ms": [_c_vp, _c_vp, _c_vp],
    "tnn_prof_enable": [_c_int],
    "tnn_prof_collect": [_c_vp, _c_vp],
    "tnn_l2_flush": [],
    "tnn_graph_begin": [],
    "tnn_graph_end": [_c_vp],
    "tnn_graph_abort": [],
    "tnn_graph_launch": [_c_vp],
    "tnn_graph_info": [_c_vp, _c_vp, _c_vp, _c_vp],
    "tnn_graph_destroy": [_c_vp],
    "tnn_ew": [_c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_int, _c_vp, _c_vp, _c_vp, _c_vp,
               _c_dbl, _c_dbl, _c_int],
    "tnn_ew_flat": [_c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_int, _c_dbl, _c_dbl,
                    _c_int],
    "tnn_cast": [_c_int, _c_vp, _c_int, _c_vp, _c_i64],
    "tnn_fill": [_c_int, _c_vp, _c_dbl, _c_i64],
    "tnn_reduce": [_c_int, _c_int, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64],
    "tnn_unbroadcast": [_c_int, _c_vp, _c_vp, _c_int, _c_vp, _c_vp],
    "tnn_strided_copy": [_c_int, _c_vp, _c_vp, _c_int, _c_vp, _c_vp, _c_vp],
    "tnn_gather_rows": [_c_int, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64],
    "tnn_scatter_rows": [_c_int, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64],
    "tnn_gather_flat": [_c_int, _c_vp, _c_vp, _c_vp, _c_i64],
    "tnn_scatter_flat": [_c_int, _c_vp, _c_vp, _c_vp, _c_i64],
    "tnn_gemm_simt": [_c_int, _c_vp, _c_i64, _c_vp, _c_i64, _c_i64, _c_vp, _c_i64, _c_i64, _c_i64,
                      _c_i64, _c_i64, _c_vp, _c_int, _c_vp, _c_vp],
    "tnn_dense_bwd_simt": [_c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_int, _c_vp, _c_int,
                           _c_i64, _c_i64, _c_i64],
    "tnn_split_tf32": [_c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_i64],
    "tnn_gemm_tf32x3": [_c_vp, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_i64, _c_i64, _c_i64,
                        _c_i64, _c_vp, _c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp],
    "tnn_split_tf32_bf16": [_c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64],
    "tnn_gemm_tf32_bf16x2": [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64,
                             _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp,
                             _c_i64, _c_vp],
    "tnn_f16_stats": [_c_vp, _c_i64, _c_vp, _c_int],
    "tnn_set_gemm_f16_cluster": [_c_int],
    "tnn_f16_meta_reset": [_c_vp],
    "tnn_split_f16": [_c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_int],
    "tnn_gemm_f16x3": [_c_vp, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64,
                       _c_i64, _c_i64, _c_vp, _c_int, _c_int, _c_vp, _c_vp, _c_vp],
    "tnn_split_tf32_bf16_cond": [_c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_int,
                                 _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_int, _c_vp, _c_vp, _c_vp],
    "tnn_f16_stats_cond": [_c_vp, _c_i64, _c_vp, _c_int],
    "tnn_gemm_tf32_bf16x2_cond": [_c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_i64,
                                  _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp],
    "tnn_set_gemm_cta_group": [_c_int],
    "tnn_set_gemm_ksplit": [_c_int],
    "tnn_set_gemm_group_m": [_c_int],
    "tnn_relu_fwd": [_c_int, _c_vp, _c_vp, _c_i64],
    "tnn_relu_bwd": [_c_int, _c_vp, _c_vp, _c_vp, _c_i64],
    "tnn_colsum": [_c_int, _c_vp, _c_vp, _c_i64, _c_i64],
    "tnn_im2col": [_c_int, _c_vp, _c_vp] + [_c_i64] * 12,
    "tnn_col2im": [_c_int, _c_vp, _c_vp] + [_c_i64] * 12,
    "tnn_maxpool_fwd": [_c_int, _c_vp, _c_vp, _c_vp] + [_c_i64] * 12,
    "tnn_maxpool_bwd": [_c_int, _c_vp, _c_vp, _c_vp] + [_c_i64] * 12,
    "tnn_bn_stats": [_c_int, _c_vp, _c_i64, _c_i64, _c_dbl, _c_dbl, _c_vp, _c_vp, _c_vp, _c_vp],
    "tnn_bn_merge": [_c_int, _c_vp, _c_int, _c_i64, _c_dbl, _c_dbl, _c_vp, _c_vp, _c_vp],
    "tnn_bn_apply": [_c_int, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_dbl],
    "tnn_bn_bwd_reduce": [_c_int, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp, _c_int, _c_vp, _c_int],
    "tnn_bn_dx": [_c_int, _c_vp, _c_vp, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_vp],
    "tnn_pointwise_loss": [_c_int, _c_int, _c_vp, _c_vp, _c_i64, _c_dbl, _c_dbl, _c_vp, _c_vp],
    "tnn_pointwise_loss_bwd": [_c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_i64, _c_dbl, _c_dbl, _c_vp],
    "tnn_ce_stats": [_c_int, _c_vp, _c_i64, _c_i64, _c_vp],
    "tnn_ce_merge_stats": [_c_int, _c_vp, _c_vp, _c_int],
    "tnn_ce_loss": [_c_int, _c_vp, _c_int, _c_vp, _c_i64, _c_i64, _c_vp, _c_dbl, _c_vp, _c_vp, _c_vp],
    "tnn_ce_fwd_small": [_c_int, _c_vp, _c_int, _c_vp, _c_i64, _c_i64, _c_dbl, _c_vp, _c_vp, _c_vp, _c_vp],
    "tnn_ce_bwd": [_c_int, _c_vp, _c_vp, _c_int, _c_vp, _c_i64, _c_i64, _c_vp, _c_vp, _c_dbl, _c_vp, _c_vp,
                   _c_vp],
    "tnn_set_gemm_reserved_sms": [_c_int],
    "tnn_d2h_async": [_c_vp, _c_vp, _c_sz, _c_vp],
    "tnn_event_sync": [_c_vp],
    "tnn_one_hot": [_c_int, _c_vp, _c_vp, _c_i64, _c_i64],
    "tnn_mlp_tail_workspace": [_c_int, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp],
    "tnn_mlp_tail_step": [_c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_int,
                          _c_i64, _c_dbl, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp],
    "tnn_opt_step": [_c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_int],
    "tnn_opt_step_dev": [_c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp],
    "tnn_nccl_unique_id": [_c_vp],
    "tnn_nccl_init": [_c_int, _c_int, _c_vp],
    "tnn_nccl_destroy": [],
    "tnn_allreduce_sum": [_c_int, _c_vp, _c_i64],
    "tnn_allgather": [_c_int, _c_vp, _c_vp, _c_i64],
    "tnn_comm_wait_compute": [],
    "tnn_compute_wait_comm": [],
    "tnn_allreduce_sum_comm": [_c_int, _c_vp, _c_i64],
    "tnn_nccl_version": [_c_vp],
}
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + ["tnn_last_error", "tnn_stream", "tnn_launch_count",
                                                "tnn_alloc_ptr"])


def load_library():
    """dlopen libtnn_b200.so and type every entry point.  Does not touch the GPU."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BackendError(
            "libtnn_b200.so not found at %s -- build it with `python tinynn-autograd_b200/build.py` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _c_int
    lib.tnn_last_error.argtypes = []
    lib.tnn_last_error.restype = ctypes.c_char_p
    lib.tnn_stream.argtypes = []
    lib.tnn_stream.restype = _c_vp
    lib.tnn_launch_count.argtypes = []
    lib.tnn_launch_count.restype = ctypes.c_uint64
    lib.tnn_alloc_ptr.argtypes = [_c_sz]
    lib.tnn_alloc_ptr.restype = _c_vp
    _lib = lib
    return lib


def _raise(name):
    msg = _lib.tnn_last_error().decode("utf-8", "replace")
    raise BackendError("%s failed: %s" % (name, msg))


def init(device=None):
    """Bind this process to one GPU.  Called lazily by the first device operation."""
    global _inited
    if _inited:
        return
    lib = load_library()
    if device is None:
        device = int(os.environ.get("TNN_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    if lib.tnn_init(int(device)):
        _raise("tnn_init")
    _inited = True


def is_initialized():
    return _inited


def sync():
    init()
    if _lib.tnn_sync():
        _raise("tnn_sync")


def launch_count():
    return int(_lib.tnn_launch_count()) if _lib is not None else 0


def device_info():
    init()
    sm, maj, mnr = _c_int(), _c_int(), _c_int()
    tot, l2 = _c_sz(), _c_sz()
    if _lib.tnn_device_info(ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr),
                            ctypes.byref(tot), ctypes.byref(l2)):
        _raise("tnn_device_info")
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "total_mem": tot.value,
            "l2_bytes": l2.value}


def set_gemm_reserved_sms(n):
    """SMs the persistent tcgen05 GEMM grid leaves free (for an NCCL kernel on the comm stream)"""
    init()
    if _lib.tnn_set_gemm_reserved_sms(int(n)):
        _raise("tnn_set_gemm_reserved_sms")


def pool_stats():
    a, b, c = _c_sz(), _c_sz(), _c_sz()
    _lib.tnn_pool_stats(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
    return {"reserved": a.value, "in_use": b.value, "cuda_mallocs": c.value}


# --------------------------------------------------------------------------------------------
# device memory
# --------------------------------------------------------------------------------------------
# Small blocks are recycled on the Python side: a freed block of a 512-byte size class is kept in a
# list and handed to the next request of that class without crossing into the library (two ctypes
# calls saved per op result; the MNIST-sized step makes ~20 such allocations and is host-bound).
# Same single-stream ordering argument as the C pool.  Blocks born inside a graph capture belong
# to that graph and never enter this cache; during a capture the cache is bypassed entirely.
_SMALL_MAX = 1 << 20          # the range the C pool rounds to 512-byte classes
_SMALL_KEEP = 64              # blocks kept per class up to 64 KiB; 8 per class above that
_SMALL_CAP_BYTES = 256 << 20  # total bytes this cache may hold back from the library's pool
_small_free = {}
_small_bytes = 0
_capturing = False


class _Buf(object):
    """Owner of one pool block; freed back to the pool when the last view dies."""
    __slots__ = ("ptr", "nbytes", "klass", "__weakref__")

    def __init__(self, nbytes):
        self.nbytes = nbytes
        if nbytes <= _SMALL_MAX and not _capturing:
            klass = (nbytes + 511) & ~511
            lst = _small_free.get(klass)
            if lst:
                global _small_bytes
                _small_bytes -= klass
                self.ptr = lst.pop()
                self.klass = klass
                return
            nbytes = klass
            self.klass = klass
        else:
            self.klass = 0
        ptr = _lib.tnn_alloc_ptr(nbytes)
        if not ptr:
            self.ptr = None
            _raise("tnn_alloc")
        self.ptr = ptr

    def __del__(self):
        try:
            ptr = self.ptr
            if not ptr or _lib is None:
                return
            if self.klass and not _capturing:
                global _small_bytes
                lst = _small_free.setdefault(self.klass, [])
                if (len(lst) < (_SMALL_KEEP if self.klass <= 65536 else 8)
                        and _small_bytes + self.klass <= _SMALL_CAP_BYTES):
                    lst.append(ptr)
                    _small_bytes += self.klass
                    return
            _lib.tnn_free(ptr)
        except Exception:
            pass


def _prod(shape):
    n = 1
    for s in shape:
        n *= s
    return n


class DArray(object):
    """Contiguous row-major device array (float32 or float64)."""
    __slots__ = ("buf", "ptr", "shape", "dtype", "size", "split", "aux", "__weakref__")

    def __init__(self, buf, ptr, shape, dtype):
        self.buf = buf
        self.ptr = ptr
        self.shape = shape
        self.dtype = dtype
        self.size = _prod(shape)
        self.split = None  # tf32 hi/lo planes cache, see split_planes()
        self.aux = None    # (pre-activation, masked gradient) left by a fused dX epilogue

    @property
    def ndim(self):
        return len(self.shape)

    @property
    def nbytes(self):
        return self.size * self.dtype.itemsize

    def view(self, shape, offset_elems=0):
        shape = tuple(int(s) for s in shape)
        return DArray(self.buf, self.ptr + offset_elems * self.dtype.itemsize, shape, self.dtype)

    def numpy(self):
        return to_numpy(self)

    def __array__(self, dtype=None, copy=None):
        a = to_numpy(self)
        return a if dtype is None else a.astype(dtype)

    def tolist(self):
        return to_numpy(self).tolist()

    def __repr__(self):
        return "DArray(shape=%s, dtype=%s)" % (self.shape, self.dtype.name)


class LazyReLU(DArray):
    """max(src, 0) that is only computed if somebody asks for its address.  The fused Dense+ReLU
    launch of the tensor-core path hands the activation on as operand planes (attached as `.split`);
    in a training step nothing reads the fp32 activation itself -- the next products use the planes,
    the backward mask uses the pre-activation -- so its 4 B/element are not written unless needed
    (`.values`, a product outside the cached step, a SIMT consumer)."""
    __slots__ = ("_src", "_real")

    def __init__(self, src):
        self._src = src
        self._real = None
        self.shape = src.shape
        self.dtype = src.dtype
        self.size = src.size
        self.split = None
        self.aux = None

    def _materialise(self):
        if self._real is None:
            self._real = relu_fwd(self._src)
        return self._real

    @property
    def ptr(self):
        return self._materialise().ptr

    @property
    def buf(self):
        return self._materialise().buf


class LazyRows(DArray):
    """src[idx[lo:hi], ...] that is only gathered when somebody asks for its address: a mini-batch of
    a shuffled epoch (utils/data_iterator.py:24-33, `inputs[idx]` then `inputs[start:end]`) named by a
    window of the epoch's permutation instead of being cut out of a shuffled copy of the data set.
    A recorded training step gathers the rows straight into its input buffer (gather_into)."""
    __slots__ = ("_src", "_idx", "_real")

    def __init__(self, src, idx_window):
        self._src = src
        self._idx = idx_window           # device int64 view, one entry per row
        self._real = None
        self.shape = (idx_window.size,) + tuple(src.shape[1:])
        self.dtype = src.dtype
        self.size = _prod(self.shape)
        self.split = None
        self.aux = None

    def gather_into(self, dst):
        """dst (same shape) <- the rows, one kernel, no intermediate"""
        assert dst.size == self.size and dst.dtype == self.dtype
        n = self.shape[0]
        row = _prod(self.shape[1:])
        if self.size and _lib.tnn_gather_rows(_DT_CODE[self.dtype], dst.ptr, self._src.ptr, self._idx.ptr, n,
                                              row, self._src.shape[0]):
            _raise("tnn_gather_rows")

    def _materialise(self):
        if self._real is None:
            self._real = gather_rows(self._src, self._idx, self.shape[0])
        return self._real

    @property
    def ptr(self):
        return self._materialise().ptr

    @property
    def buf(self):
        return self._materialise().buf

    def view(self, shape, offset_elems=0):
        return self._materialise().view(shape, offset_elems)


class LazyOneHot(DArray):
    """(n, C) float32 one-hot rows named by n int32 class indices on the device; written
    (tnn_one_hot, run.py:27-28 get_one_hot) only if somebody asks for their address.  The fused
    cross-entropy takes the indices themselves (ops.softmax_ce_), so in a training step fed by
    utils.data_iterator.PrefetchIterator the dense label matrix -- 134 MB per batch for the wide
    MLP -- is neither written nor read."""
    __slots__ = ("_labels", "_dst", "_real")

    def __init__(self, labels, n_classes, dst):
        self._labels = labels            # device vector of n int32 indices (kept in a 4-byte float view)
        self._dst = dst                  # (n, C) float32 array that receives the rows on demand
        self._real = None
        self.shape = (labels.shape[0], int(n_classes))
        self.dtype = F32
        self.size = _prod(self.shape)
        self.split = None
        self.aux = None

    def _materialise(self):
        if self._real is None:
            one_hot_into(self._dst, self._labels.ptr, self.shape[0], self.shape[1])
            self._real = self._dst
        return self._real

    @property
    def labels_ptr(self):
        return self._labels.ptr

    @property
    def ptr(self):
        return self._materialise().ptr

    @property
    def buf(self):
        return self._materialise().buf

    def view(self, shape, offset_elems=0):
        return self._materialise().view(shape, offset_elems)


def device_dtype(np_dtype):
    """dtype policy: float32 stays float32; everything else (ints, bools, float64, Python
    numbers) is computed in float64 so the reference's exact-equality tests hold (SURVEY Q7/Q8)."""
    dt = np.dtype(np_dtype)
    if dt == F32 or dt == np.float16:
        return F32
    if dt.kind in "fiub":
        return F64
    raise TypeError("unsupported dtype for a device tensor: %s" % dt)


def empty(shape, dtype):
    if not _inited:
        init()
    if type(shape) is not tuple:
        shape = tuple(int(s) for s in shape)
    if type(dtype) is not np.dtype:
        dtype = np.dtype(dtype)
    n = 1
    for s in shape:
        n *= s
    buf = _Buf((n if n > 0 else 1) * dtype.itemsize)
    return DArray(buf, buf.ptr, shape, dtype)


def from_numpy(arr, dtype=None):
    arr = np.asarray(arr)
    dt = device_dtype(arr.dtype if dtype is None else dtype)
    host = np.require(arr, dtype=dt, requirements="C")  # (ascontiguousarray would make 0-d 1-d)
    out = empty(host.shape, dt)
    if host.size:
        if _lib.tnn_h2d(out.ptr, host.ctypes.data, host.nbytes):
            _raise("tnn_h2d")
    return out


def upload_into(dst, host):
    """host array -> existing device array (same dtype and element count)"""
    host = np.require(host, dtype=dst.dtype, requirements="C")
    assert host.size == dst.size
    if host.size and _lib.tnn_h2d(dst.ptr, host.ctypes.data, host.nbytes):
        _raise("tnn_h2d")


def to_numpy(d):
    out = np.empty(d.shape, dtype=d.dtype)
    if d.size:
        if _lib.tnn_d2h(out.ctypes.data, d.ptr, out.nbytes):
            _raise("tnn_d2h")
    return out


def full(shape, value, dtype):
    out = empty(shape, dtype)
    if out.size:
        if _lib.tnn_fill(_DT_CODE[out.dtype], out.ptr, float(value), out.size):
            _raise("tnn_fill")
    return out


_ONES = {}


def ones_scalar(dtype):
    """a persistent 0-d array holding 1.0 (the default seed of backward()); never written again"""
    dtype = np.dtype(dtype)
    one = _ONES.get(dtype)
    if one is None:
        one = _ONES[dtype] = full((), 1.0, dtype)
    return one


def zeros(shape, dtype):
    out = empty(shape, dtype)
    if out.size:
        if _lib.tnn_memset(out.ptr, 0, out.nbytes):
            _raise("tnn_memset")
    return out


def memset_zero(d):
    if d.size and _lib.tnn_memset(d.ptr, 0, d.nbytes):
        _raise("tnn_memset")


def copy_into(dst, src):
    assert dst.size == src.size and dst.dtype == src.dtype
    if dst.size and _lib.tnn_d2d(dst.ptr, src.ptr, dst.nbytes):
        _raise("tnn_d2d")


def clone(d):
    out = empty(d.shape, d.dtype)
    copy_into(out, d)
    return out


def astype(d, dtype):
    dtype = np.dtype(dtype)
    if d.dtype == dtype:
        return d
    out = empty(d.shape, dtype)
    if d.size and _lib.tnn_cast(_DT_CODE[dtype], out.ptr, _DT_CODE[d.dtype], d.ptr, d.size):
        _raise("tnn_cast")
    return out


def upload_index(idx):
    """int64 index vector -> raw device buffer (returned as a DArray typed float64 only for
    bookkeeping; kernels read it as int64)."""
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    out = empty(idx.shape, F64)
    if idx.size and _lib.tnn_h2d(out.ptr, idx.ctypes.data, idx.nbytes):
        _raise("tnn_h2d")
    return out


# --------------------------------------------------------------------------------------------
# elementwise
# --------------------------------------------------------------------------------------------
def _i64arr(vals):
    return (_c_i64 * len(vals))(*vals)


def _bstrides(shape, out_shape):
    """element strides of a contiguous `shape` array broadcast (numpy rules) to out_shape"""
    nd = len(out_shape)
    pad = nd - len(shape)
    st = [0] * nd
    acc = 1
    for i in range(len(shape) - 1, -1, -1):
        if shape[i] != 1:
            st[pad + i] = acc
        acc *= shape[i]
    return st


def _common_dtype(*arrs):
    for a in arrs:
        if a.dtype == F64:
            return F64
    return F32


def ew(op, x, y=None, z=None, p0=0.0, p1=0.0, flags=0, out=None):
    """out = op(x, y, z) with numpy broadcasting; operands are promoted to a common dtype."""
    ops_ = [a for a in (x, y, z) if a is not None]
    dt = _common_dtype(*ops_)
    ops_ = [a if a.dtype == dt else astype(a, dt) for a in ops_]
    if len(ops_) == 1:
        oshape = ops_[0].shape
    else:
        oshape = ops_[0].shape
        for a in ops_[1:]:
            if a.shape != oshape:
                oshape = np.broadcast_shapes(*[a.shape for a in ops_])  # ValueError like numpy
                break
    if out is None:
        out = empty(oshape, dt)
    n = out.size
    if n == 0:
        return out
    ptrs = [a.ptr for a in ops_] + [None] * (3 - len(ops_))
    mask = 0
    flat = True
    for i, a in enumerate(ops_):
        if a.size == 1:
            mask |= 1 << i
        elif a.shape != oshape:
            # same element count and layout (e.g. (3,) vs (1,3)) still counts as flat
            if a.size == n and _bstrides(a.shape, oshape) == _bstrides(oshape, oshape):
                continue
            flat = False
    if flat:
        if _lib.tnn_ew_flat(op, _DT_CODE[dt], out.ptr, ptrs[0], ptrs[1], ptrs[2], n, mask,
                            p0, p1, flags):
            _raise("tnn_ew_flat")
        return out
    nd = len(oshape)
    if nd > MAX_DIMS:
        raise ValueError("tensors of rank > %d are not supported" % MAX_DIMS)
    st = [_i64arr(_bstrides(a.shape, oshape)) for a in ops_] + [None] * (3 - len(ops_))
    if _lib.tnn_ew(op, _DT_CODE[dt], out.ptr, ptrs[0], ptrs[1], ptrs[2], nd, _i64arr(oshape),
                   st[0], st[1], st[2], p0, p1, flags):
        _raise("tnn_ew")
    return out


def add_inplace(dst, src):
    """dst += src (same shape, same dtype)"""
    if src.dtype != dst.dtype:
        src = astype(src, dst.dtype)
    if _lib.tnn_ew_flat(ADD, _DT_CODE[dst.dtype], dst.ptr, dst.ptr, src.ptr, None, dst.size,
                        2 if (src.size == 1 and dst.size != 1) else 0, 0.0, 0.0, 0):
        _raise("tnn_ew_flat")
    return dst


def broadcast_to(d, shape):
    shape = tuple(shape)
    if d.shape == shape:
        return d
    out = empty(shape, d.dtype)
    oshape = np.broadcast_shapes(d.shape, shape)
    if tuple(oshape) != shape:
        raise ValueError("cannot broadcast %s to %s" % (d.shape, shape))
    if out.size:
        if _lib.tnn_ew(COPY, _DT_CODE[d.dtype], out.ptr, d.ptr, None, None, len(shape),
                       _i64arr(shape), _i64arr(_bstrides(d.shape, shape)), None, None, 0.0, 0.0, 0):
            _raise("tnn_ew")
    return out


# --------------------------------------------------------------------------------------------
# reductions / unbroadcast
# --------------------------------------------------------------------------------------------
def reduce(red_op, x, axis=None):
    """np.sum / np.max / np.min with axis=None or an int (ops.py:225-265)"""
    if axis is None:
        outer, red, inner = 1, x.size, 1
        oshape = ()
    else:
        nd = x.ndim
        if not -nd <= axis < nd:
            raise np.exceptions.AxisError(axis, nd)
        axis %= nd
        outer = _prod(x.shape[:axis])
        red = x.shape[axis]
        inner = _prod(x.shape[axis + 1:])
        oshape = x.shape[:axis] + x.shape[axis + 1:]
    if red == 0 and red_op != RED_SUM:
        raise ValueError("zero-size array to reduction operation which has no identity")
    out = empty(oshape, x.dtype)
    if out.size:
        if _lib.tnn_reduce(red_op, _DT_CODE[x.dtype], out.ptr, x.ptr, outer, red, inner):
            _raise("tnn_reduce")
    return out


def unbroadcast(g, shape):
    """Sum g down to `shape` exactly as the loops at ops.py:41-46 do."""
    shape = tuple(shape)
    if g.shape == shape:
        return g
    nd = g.ndim
    lead = nd - len(shape)
    if lead < 0:
        raise ValueError("gradient of rank %d for a tensor of rank %d" % (nd, len(shape)))
    keep = [0] * lead + [0 if s == 1 else 1 for s in shape]
    for i in range(len(shape)):
        if shape[i] != 1 and shape[i] != g.shape[lead + i]:
            raise ValueError("operands could not be broadcast together with shapes %s %s"
                             % (g.shape, shape))
    out = empty(shape, g.dtype)
    if out.size:
        if _lib.tnn_unbroadcast(_DT_CODE[g.dtype], out.ptr, g.ptr, nd, _i64arr(g.shape),
                                (_c_i32 * nd)(*keep)):
            _raise("tnn_unbroadcast")
    return out


def colsum(g, out=None):
    """(R, C) -> (1, C): the bias gradient"""
    R, C = g.shape
    if out is None:
        out = empty((1, C), g.dtype)
    if _lib.tnn_colsum(_DT_CODE[g.dtype], out.ptr, g.ptr, R, C):
        _raise("tnn_colsum")
    return out


# --------------------------------------------------------------------------------------------
# layout
# --------------------------------------------------------------------------------------------
def _cstrides(shape):
    st = [0] * len(shape)
    acc = 1
    for i in range(len(shape) - 1, -1, -1):
        st[i] = acc
        acc *= shape[i]
    return st


def permute(x, axes):
    nd = x.ndim
    axes = [a % nd for a in axes]
    oshape = tuple(x.shape[a] for a in axes)
    out = empty(oshape, x.dtype)
    if out.size:
        xs = _cstrides(x.shape)
        if _lib.tnn_strided_copy(_DT_CODE[x.dtype], out.ptr, x.ptr, nd, _i64arr(oshape),
                                 _i64arr(_cstrides(oshape)), _i64arr([xs[a] for a in axes])):
            _raise("tnn_strided_copy")
    return out


def strided_copy(dst, dst_off, dst_strides, src, src_off, src_strides, shape):
    if _prod(shape) == 0:
        return
    isz = dst.dtype.itemsize
    if _lib.tnn_strided_copy(_DT_CODE[dst.dtype], dst.ptr + dst_off * isz, src.ptr + src_off * isz,
                             len(shape), _i64arr(shape), _i64arr(dst_strides), _i64arr(src_strides)):
        _raise("tnn_strided_copy")


def one_hot_into(out, labels_i32_ptr, n_rows, n_classes):
    """out (n_rows, n_classes) <- one-hot rows of the int32 device vector at `labels_i32_ptr`"""
    if _lib.tnn_one_hot(_DT_CODE[out.dtype], out.ptr, labels_i32_ptr, n_rows, n_classes):
        _raise("tnn_one_hot")


def gather_rows(x, idx_dev, n_idx):
    row = _prod(x.shape[1:])
    out = empty((n_idx,) + x.shape[1:], x.dtype)
    if out.size and _lib.tnn_gather_rows(_DT_CODE[x.dtype], out.ptr, x.ptr, idx_dev.ptr, n_idx, row,
                                         x.shape[0]):
        _raise("tnn_gather_rows")
    return out


def scatter_rows(g, idx_dev, n_idx, shape):
    out = zeros(shape, g.dtype)
    row = _prod(shape[1:])
    if g.size and _lib.tnn_scatter_rows(_DT_CODE[g.dtype], out.ptr, g.ptr, idx_dev.ptr, n_idx, row,
                                        shape[0]):
        _raise("tnn_scatter_rows")
    return out


def gather_flat(x, idx_dev, oshape):
    out = empty(oshape, x.dtype)
    if out.size and _lib.tnn_gather_flat(_DT_CODE[x.dtype], out.ptr, x.ptr, idx_dev.ptr, out.size):
        _raise("tnn_gather_flat")
    return out


def scatter_flat(g, idx_dev, shape):
    out = zeros(shape, g.dtype)
    if g.size and _lib.tnn_scatter_flat(_DT_CODE[g.dtype], out.ptr, g.ptr, idx_dev.ptr, g.size):
        _raise("tnn_scatter_flat")
    return out


# --------------------------------------------------------------------------------------------
# GEMM
# --------------------------------------------------------------------------------------------
# below this M*N*K the SIMT kernel is at least as fast as the tensor-core path with its operand
# passes (statistics, split, product, two conditional launches: ~58 us of launches for fresh operands
# against 13-54 us of SIMT GEMM up to 2^29; scripts/tc_threshold.py, profiles/r02f_tc_threshold.txt)
TC_MIN_MNK = int(os.environ.get("TNN_TC_MIN_MNK", str(1 << 29)))
TC_ENABLED = os.environ.get("TNN_TC", "1") != "0"
TC_MN_MAJOR = os.environ.get("TNN_TC_MN_MAJOR", "1") != "0"   # 0: transposed tf32 planes instead
# operand split of the tensor-core product: "mix" = tf32 main term + bf16 cross terms (default),
# "tf32x3" = three tf32 MMAs per K step (the textbook 3xTF32, kept as cross-check)
# "f16" (default) = scaled fp16 + bf16 planes, three kind::f16 MMAs (gemm_f16.cu), with the mixed
# split as on-device fallback for operands outside its guard;
TC_SPLIT = os.environ.get("TNN_GEMM_SPLIT", "f16")
# fused Dense+ReLU launch on the tensor-core path: do not write the fp32 activation (see LazyReLU)
LAZY_RELU_OUT = os.environ.get("TNN_LAZY_RELU", "1") != "0"
BF16_BYTES = 2
_split_epoch = 0


def new_split_epoch():
    """Called once per training step: tf32 planes of activations never outlive a step."""
    global _split_epoch
    _split_epoch += 1


def _round4(n):
    return (n + 3) // 4 * 4


def _round8(n):
    return (n + 7) // 8 * 8


def _empty_16bit(rows, ld):
    """raw 16-bit plane, bf16 or fp16 (kept as a float32 DArray of half the width for bookkeeping)"""
    return empty((rows, ld // 2), F32)


def _plane_cache(x):
    """x's operand-plane cache for the current step (a fresh one when x has none from this step)"""
    cache = x.split
    if cache is None or cache.get("epoch") != _split_epoch:
        cache = {"epoch": _split_epoch}
        x.split = cache
    return cache


def split_planes_mix(x):
    """fp32 (R, C) -> (hi tf32 plane, bf16(x), bf16(x - hi), ld), cached for the step"""
    cache = _plane_cache(x)
    if "m" in cache:
        return cache["m"]
    R, C = x.shape
    ld = _round8(C)
    hi, h16, l16 = empty((R, ld), F32), _empty_16bit(R, ld), _empty_16bit(R, ld)
    if _lib.tnn_split_tf32_bf16(x.ptr, R, C, hi.ptr, h16.ptr, l16.ptr, ld):
        _raise("tnn_split_tf32_bf16")
    cache["m"] = (hi, h16, l16, ld)
    return cache["m"]


F16_PITCH_PAD = int(os.environ.get("TNN_F16_PITCH_PAD", "0"))   # extra plane pitch, multiple of 8 elements


def _new_meta():
    """32-byte operand record of the f16 split (gemm_f16.cu: Meta)"""
    return empty((8,), F32)


def split_planes_f16(x):
    """fp32 (R, C) -> (hf fp16 plane, l16 bf16 plane, ld, meta, source array, relu_mode), cached for
    the step.  A LazyReLU is split straight from its pre-activation (relu applied on load); the
    statistics come from the producer's epilogue when it left a record (cache["stat"])."""
    cache = _plane_cache(x)
    if "f" in cache:
        return cache["f"]
    R, C = x.shape
    ld = _round8(C) + F16_PITCH_PAD
    if type(x) is LazyReLU and x._real is None:
        src, relu_mode = x._src, 1
    else:
        src, relu_mode = x, 0
    meta = cache.get("stat")
    if meta is None:
        meta = _new_meta()
        if _lib.tnn_f16_stats(src.ptr, R * C, meta.ptr, relu_mode):
            _raise("tnn_f16_stats")
    elif _lib.tnn_f16_stats_cond(src.ptr, R * C, meta.ptr, relu_mode):
        # (the producer's epilogue normally recorded them; this launch only works when the producer
        # was the fallback product, which records none)
        _raise("tnn_f16_stats_cond")
    hf, l16 = _empty_16bit(R, ld), _empty_16bit(R, ld)
    if _lib.tnn_split_f16(src.ptr, R, C, hf.ptr, l16.ptr, ld, meta.ptr, relu_mode):
        _raise("tnn_split_f16")
    # (the source is not stored when it is x itself: x -> x.split -> x would be a reference cycle,
    # and blocks held by cycles are only returned to the pool by the garbage collector)
    cache["f"] = (hf, l16, ld, meta, src if src is not x else None, relu_mode)
    return cache["f"]


_FALLBACK_PLANES = {}
_FALLBACK_CAP_BYTES = 16 << 30     # many distinct product shapes in one process: start over past this
_fallback_bytes = 0


def _fallback_planes(role, R, ld):
    """scratch for the conditional mixed split behind an f16 product.  Outside a capture: one set per
    (role, shape), reused by every later product of that shape (same stream: ordered) and never
    returned to the pool, so nothing that was enqueued can find it recycled under it.  While a step is
    being recorded the planes are fresh blocks, which belong to the graph until it is destroyed (a
    recorded conditional split must not point at scratch that eager products also use)."""
    if _capturing:
        return (empty((R, ld), F32), _empty_16bit(R, ld), _empty_16bit(R, ld))
    global _fallback_bytes
    key = (role, R, ld)
    p = _FALLBACK_PLANES.get(key)
    if p is None:
        if _fallback_bytes > _FALLBACK_CAP_BYTES:
            sync()                       # nothing enqueued points at the old sets any more
            _FALLBACK_PLANES.clear()
            _fallback_bytes = 0
        p = (empty((R, ld), F32), _empty_16bit(R, ld), _empty_16bit(R, ld))
        _FALLBACK_PLANES[key] = p
        _fallback_bytes += 8 * R * ld
    return p


def _matmul_f16(a, b, ta, tb, bias, out, flags, act, mask_src, M, N, K):
    a_hf, a_l16, lda, a_meta, a_src, a_relu = split_planes_f16(a)
    b_hf, b_l16, ldb, b_meta, b_src, b_relu = split_planes_f16(b)
    a_src = a if a_src is None else a_src
    b_src = b if b_src is None else b_src
    layout = (1 if ta else 0) | (0 if tb else 2)
    act_out = None
    stat = None
    if act:
        stat = _new_meta()
        if _lib.tnn_f16_meta_reset(stat.ptr):
            _raise("tnn_f16_meta_reset")
        if mask_src is None and LAZY_RELU_OUT:
            act_out = LazyReLU(out)          # statistics only: the fp32 activation is not written
            flags |= 8
        else:
            act_out = empty((M, N), F32)
    real_act = act_out if (act and type(act_out) is not LazyReLU) else None
    bias_p = bias.ptr if bias is not None else None
    mask_p = mask_src.ptr if (act and mask_src is not None) else None
    if _lib.tnn_gemm_f16x3(out.ptr, N, a_hf.ptr, a_l16.ptr, lda, a_meta.ptr, b_hf.ptr, b_l16.ptr, ldb,
                           b_meta.ptr, M, N, K, bias_p, flags, layout,
                           real_act.ptr if real_act is not None else None, mask_p,
                           stat.ptr if stat is not None else None):
        _raise("tnn_gemm_f16x3")
    # on-device fallback: these three launches return at once when both operands were inside the guard
    fa = _fallback_planes(0, a.shape[0], lda)
    fb = _fallback_planes(1, b.shape[0], ldb)
    if _lib.tnn_split_tf32_bf16_cond(a_src.ptr, a.shape[0], a.shape[1], fa[0].ptr, fa[1].ptr, fa[2].ptr, lda,
                                     a_relu, b_src.ptr, b.shape[0], b.shape[1], fb[0].ptr, fb[1].ptr,
                                     fb[2].ptr, ldb, b_relu, a_meta.ptr, b_meta.ptr,
                                     stat.ptr if stat is not None else None):
        _raise("tnn_split_tf32_bf16_cond")
    if _lib.tnn_gemm_tf32_bf16x2_cond(out.ptr, N, fa[0].ptr, fa[1].ptr, fa[2].ptr, lda, fb[0].ptr, fb[1].ptr,
                                      fb[2].ptr, ldb, M, N, K, bias_p, flags & 3, layout,
                                      real_act.ptr if real_act is not None else None, mask_p,
                                      a_meta.ptr, b_meta.ptr):
        _raise("tnn_gemm_tf32_bf16x2_cond")
    if act:
        act_out.split = {"epoch": _split_epoch, "stat": stat}
        return out, act_out
    return out


def split_planes(x, transposed, also_other=False):
    """fp32 (R, C) -> tf32 (hi, lo, ld) planes; transposed=True gives the (C, R) planes.
    Planes are cached on the array for the current step so forward and backward share them."""
    cache = _plane_cache(x)
    key = "t" if transposed else "p"
    if key in cache:
        return cache[key]
    R, C = x.shape
    want_p = (not transposed) or (also_other and "p" not in cache)
    want_t = transposed or (also_other and "t" not in cache)
    hi = lo = hit = lot = None
    ldp = _round4(C)
    ldt = _round4(R)
    if want_p:
        hi, lo = empty((R, ldp), F32), empty((R, ldp), F32)
    if want_t:
        hit, lot = empty((C, ldt), F32), empty((C, ldt), F32)
    if _lib.tnn_split_tf32(x.ptr, R, C, hi.ptr if hi else None, lo.ptr if lo else None, ldp,
                           hit.ptr if hit else None, lot.ptr if lot else None, ldt):
        _raise("tnn_split_tf32")
    if want_p:
        cache["p"] = (hi, lo, ldp)
    if want_t:
        cache["t"] = (hit, lot, ldt)
    return cache[key]


def set_gemm_cta_group(cg):
    load_library()
    if _lib.tnn_set_gemm_cta_group(int(cg)):
        _raise("tnn_set_gemm_cta_group")


def set_gemm_f16_cluster(cl):
    load_library()
    if _lib.tnn_set_gemm_f16_cluster(int(cl)):
        _raise("tnn_set_gemm_f16_cluster")


def set_gemm_ksplit(ks):
    load_library()
    if _lib.tnn_set_gemm_ksplit(int(ks)):
        _raise("tnn_set_gemm_ksplit")


def use_tensor_cores(M, N, K, dtype):
    return (TC_ENABLED and dtype == F32 and M >= 64 and N >= 64 and K >= 32
            and M * N * K >= TC_MIN_MNK)


def matmul(a, b, ta=False, tb=False, bias=None, out=None, accumulate=False, relu=False,
           reuse_a=False, reuse_b=False, act=False, mask_src=None):
    """op(a) @ op(b) (+ bias) for 2-D arrays; op = transpose when ta/tb (ops.py:150-160).

    float32 products above TC_MIN_MNK run on a tcgen05 tensor-core kernel chosen by TC_SPLIT: the
    scaled fp16 split by default (with the mixed split as its on-device fallback), the mixed
    tf32/bf16 split, or 3xTF32; float64 and small or odd-shaped products run on the SIMT kernel.
    reuse_a/reuse_b hint that the other orientation of that operand will be needed later in the
    step (forward -> backward), so both sets of 3xTF32 planes are produced by one pass.

    act=True returns (out, relu(out)): the GEMM epilogue writes the ReLU of its result as a second
    array -- and, on the tensor-core path, that array's tf32 planes, which are attached to it so the
    next product consumes it without a separate ReLU or split pass.  With mask_src (the
    pre-activation of the ReLU that produced op(b)'s counterpart) the second array is instead
    out * (mask_src >= 0): the ReLU backward fused into the dX product."""
    if a.ndim != 2 or b.ndim != 2:
        raise ValueError("matmul: only 2-D operands are supported (got %s @ %s)" % (a.shape, b.shape))
    dt = _common_dtype(a, b)
    if a.dtype != dt:
        a = astype(a, dt)
    if b.dtype != dt:
        b = astype(b, dt)
    M, K = (a.shape[1], a.shape[0]) if ta else a.shape
    K2, N = (b.shape[1], b.shape[0]) if tb else b.shape
    if K != K2:
        raise ValueError("matmul: shapes %s and %s not aligned" % ((M, K), (K2, N)))
    if out is None:
        out = empty((M, N), dt)
        accumulate = False
    elif out.dtype != dt or out.shape != (M, N):
        raise ValueError("matmul: bad output array")
    if bias is not None and bias.dtype != dt:
        bias = astype(bias, dt)
    act_out = empty((M, N), dt) if act else None
    if M == 0 or N == 0:
        return (out, act_out) if act else out
    flags = (1 if accumulate else 0) | (2 if relu else 0)
    if K > 0 and use_tensor_cores(M, N, K, dt) and TC_SPLIT == "f16":
        return _matmul_f16(a, b, ta, tb, bias, out, flags, act, mask_src, M, N, K)
    if K > 0 and use_tensor_cores(M, N, K, dt) and TC_SPLIT == "mix":
        a_hi, a_h16, a_l16, lda = split_planes_mix(a)
        b_hi, b_h16, b_l16, ldb = split_planes_mix(b)
        layout = (1 if ta else 0) | (0 if tb else 2)
        act_hi = act_h16 = act_l16 = None
        ld_act = _round8(N)
        if act:
            act_hi = empty((M, ld_act), F32)
            act_h16, act_l16 = _empty_16bit(M, ld_act), _empty_16bit(M, ld_act)
            if LAZY_RELU_OUT and mask_src is None:
                act_out = LazyReLU(out)      # planes only: the fp32 activation is not written
        if _lib.tnn_gemm_tf32_bf16x2(out.ptr, N, a_hi.ptr, a_h16.ptr, a_l16.ptr, lda, b_hi.ptr,
                                     b_h16.ptr, b_l16.ptr, ldb, M, N, K,
                                     bias.ptr if bias is not None else None, flags, layout,
                                     act_out.ptr if (act and type(act_out) is not LazyReLU) else None,
                                     act_hi.ptr if act else None,
                                     act_h16.ptr if act else None, act_l16.ptr if act else None,
                                     ld_act, mask_src.ptr if (act and mask_src is not None) else None):
            _raise("tnn_gemm_tf32_bf16x2")
        if act:
            act_out.split = {"epoch": _split_epoch, "m": (act_hi, act_h16, act_l16, ld_act)}
            return out, act_out
        return out
    if K > 0 and use_tensor_cores(M, N, K, dt):
        if TC_MN_MAJOR:
            # un-transposed planes only: a transposed operand is fed MN-major to the tensor core
            a_hi, a_lo, lda = split_planes(a, transposed=False)
            b_hi, b_lo, ldb = split_planes(b, transposed=False)
            layout = (1 if ta else 0) | (0 if tb else 2)
        else:
            a_hi, a_lo, lda = split_planes(a, transposed=ta, also_other=reuse_a)
            b_hi, b_lo, ldb = split_planes(b, transposed=not tb, also_other=reuse_b)
            layout = 0
        act_hi = act_lo = None
        ld_act = _round4(N)
        if act:
            act_hi, act_lo = empty((M, ld_act), F32), empty((M, ld_act), F32)
        if _lib.tnn_gemm_tf32x3(out.ptr, N, a_hi.ptr, a_lo.ptr, lda, b_hi.ptr, b_lo.ptr, ldb, M, N,
                                K, bias.ptr if bias is not None else None, flags, layout,
                                act_out.ptr if act else None, act_hi.ptr if act else None,
                                act_lo.ptr if act else None, ld_act,
                                mask_src.ptr if (act and mask_src is not None) else None):
            _raise("tnn_gemm_tf32x3")
        if act:
            act_out.split = {"epoch": _split_epoch, "p": (act_hi, act_lo, ld_act)}
            return out, act_out
        return out
    a_rs, a_cs = (1, a.shape[1]) if ta else (a.shape[1], 1)
    b_rs, b_cs = (1, b.shape[1]) if tb else (b.shape[1], 1)
    if mask_src is not None and mask_src.dtype != dt:
        mask_src = astype(mask_src, dt)
    if _lib.tnn_gemm_simt(_DT_CODE[dt], out.ptr, N, a.ptr, a_rs, a_cs, b.ptr, b_rs, b_cs, M, N, K,
                          bias.ptr if bias is not None else None, flags & 1,
                          act_out.ptr if act else None,
                          mask_src.ptr if (act and mask_src is not None) else None):
        _raise("tnn_gemm_simt")
    if relu:
        if _lib.tnn_relu_fwd(_DT_CODE[dt], out.ptr, out.ptr, out.size):
            _raise("tnn_relu_fwd")
    return (out, act_out) if act else out


GROUPED_BWD_MAX_TILES = 1024   # above this the three products are big enough to launch on their own


def dense_bwd_grouped_ok(B, K, N, dtype):
    """small Dense layer: its three gradient products go out as one grouped SIMT launch"""
    if use_tensor_cores(B, K, N, dtype) or use_tensor_cores(K, N, B, dtype):
        return False
    t = lambda m, n: ((m + 31) // 32) * ((n + 31) // 32)
    return t(K, N) + t(B, K) + t(1, N) <= GROUPED_BWD_MAX_TILES


def dense_bwd_grouped(g, x, w, mask_src, need_dx, dw_out, dw_acc, db_out, db_acc):
    """(dx, dx_masked) -- either may be None -- with dW / db written (or accumulated) in place"""
    B, N = g.shape
    K = w.shape[0]
    dx = empty((B, K), g.dtype) if need_dx else None
    masked = empty((B, K), g.dtype) if (need_dx and mask_src is not None) else None
    if _lib.tnn_dense_bwd_simt(_DT_CODE[g.dtype], g.ptr, x.ptr, w.ptr,
                               mask_src.ptr if masked is not None else None,
                               dx.ptr if dx is not None else None,
                               masked.ptr if masked is not None else None,
                               dw_out.ptr, 1 if dw_acc else 0, db_out.ptr, 1 if db_acc else 0, B, K, N):
        _raise("tnn_dense_bwd_simt")
    return dx, masked


# --------------------------------------------------------------------------------------------
# fused layer / loss / optimizer kernels
# --------------------------------------------------------------------------------------------
def relu_fwd(x):
    out = empty(x.shape, x.dtype)
    if x.size and _lib.tnn_relu_fwd(_DT_CODE[x.dtype], out.ptr, x.ptr, x.size):
        _raise("tnn_relu_fwd")
    return out


def relu_bwd(g, x):
    if g.dtype != x.dtype:
        g = astype(g, x.dtype)
    out = empty(x.shape, x.dtype)
    if x.size and _lib.tnn_relu_bwd(_DT_CODE[x.dtype], out.ptr, g.ptr, x.ptr, x.size):
        _raise("tnn_relu_bwd")
    return out


# NHWC window passes (csrc/conv.cu).  `geom` = (KH, KW, SH, SW, PH0, PW0, OH, OW): window, stride,
# padding before the first row / column and output extent, as core.layers.window_geometry gives them.
def im2col(x, geom):
    """(N, H, W, C) -> col (N*OH*OW, KH*KW*C), zeros where a window reaches into the padding"""
    N, H, W, C = x.shape
    KH, KW, _, _, _, _, OH, OW = geom
    out = empty((N * OH * OW, KH * KW * C), x.dtype)
    if out.size and _lib.tnn_im2col(_DT_CODE[x.dtype], out.ptr, x.ptr, N, H, W, C, *geom):
        _raise("tnn_im2col")
    return out


def col2im(dcol, x_shape, geom):
    """adjoint of im2col: dx of shape x_shape, each element the sum of the dcol entries that read it"""
    N, H, W, C = x_shape
    out = empty(x_shape, dcol.dtype)
    if out.size and _lib.tnn_col2im(_DT_CODE[dcol.dtype], out.ptr, dcol.ptr, N, H, W, C, *geom):
        _raise("tnn_col2im")
    return out


def maxpool_fwd(x, geom):
    """(y, arg): the window maxima (N, OH, OW, C) and, as int32, each one's offset in its window"""
    N, H, W, C = x.shape
    OH, OW = geom[6], geom[7]
    y = empty((N, OH, OW, C), x.dtype)
    arg = empty((N, OH, OW, C), np.int32)
    if y.size and _lib.tnn_maxpool_fwd(_DT_CODE[x.dtype], y.ptr, arg.ptr, x.ptr, N, H, W, C, *geom):
        _raise("tnn_maxpool_fwd")
    return y, arg


def maxpool_bwd(g, arg, x_shape, geom):
    """dx of shape x_shape: each element sums the gradients of the windows that selected it"""
    N, H, W, C = x_shape
    out = empty(x_shape, g.dtype)
    if out.size and _lib.tnn_maxpool_bwd(_DT_CODE[g.dtype], out.ptr, g.ptr, arg.ptr, N, H, W, C, *geom):
        _raise("tnn_maxpool_bwd")
    return out


# Batch normalisation passes (csrc/batchnorm.cu) on an (M, C) view.  `mr` is the (2C + 1,) float64
# array of column means, r = 1/sqrt(var + eps) and the row count the statistics cover.
def bn_stats(x, momentum, eps, running_mean, running_var, local=False):
    """TRAIN statistics of x (M, C): mr, with the running statistics updated in place -- or, with
    `local`, this rank's (M, mean[C], M2[C]) as a (1 + 2C,) float64 array and nothing updated"""
    M, C = x.shape
    out = empty((1 + 2 * C,) if local else (2 * C + 1,), F64)
    mr, part = (None, out.ptr) if local else (out.ptr, None)
    if _lib.tnn_bn_stats(_DT_CODE[x.dtype], x.ptr, M, C, float(momentum), float(eps), running_mean.ptr,
                         running_var.ptr, mr, part):
        _raise("tnn_bn_stats")
    return out


def bn_merge(gathered, world, C, momentum, eps, running_mean, running_var):
    """`world` ranks' local statistics (bn_stats(local=True), gathered in rank order) -> mr, with the
    running statistics updated in place"""
    mr = empty((2 * C + 1,), F64)
    if _lib.tnn_bn_merge(_DT_CODE[running_mean.dtype], gathered.ptr, world, C, float(momentum), float(eps),
                         running_mean.ptr, running_var.ptr, mr.ptr):
        _raise("tnn_bn_merge")
    return mr


def bn_apply(x, gamma, beta, mr=None, running=None, eps=0.0):
    """(y, mr): y = (x - mean) * r * gamma + beta with the statistics of mr (TRAIN) or, given
    running = (running_mean, running_var), of the running statistics (TEST; mr is then made here)"""
    M, C = x.shape
    y = empty((M, C), x.dtype)
    if running is not None:
        mr = empty((2 * C + 1,), F64)
    rm, rv = (running[0].ptr, running[1].ptr) if running is not None else (None, None)
    if _lib.tnn_bn_apply(_DT_CODE[x.dtype], y.ptr, x.ptr, M, C, gamma.ptr, beta.ptr, mr.ptr, rm, rv, float(eps)):
        _raise("tnn_bn_apply")
    return y, mr


def bn_bwd_reduce(g, x, mr, dgamma, acc_gamma, dbeta, acc_beta):
    """(sum dy, sum dy * xhat) per column as one (2C,) float64 array; dbeta / dgamma (C values each,
    or None) receive the two halves, written or (acc_*) added"""
    M, C = x.shape
    sums = empty((2 * C,), F64)
    if _lib.tnn_bn_bwd_reduce(_DT_CODE[x.dtype], g.ptr, x.ptr, M, C, mr.ptr, sums.ptr,
                              dgamma.ptr if dgamma is not None else None, int(acc_gamma),
                              dbeta.ptr if dbeta is not None else None, int(acc_beta)):
        _raise("tnn_bn_bwd_reduce")
    return sums


def bn_dx(g, x, mr, gamma, sums=None):
    """dx of the normalisation: with the batch statistics' terms when `sums` is given (TRAIN)"""
    M, C = x.shape
    dx = empty((M, C), x.dtype)
    if _lib.tnn_bn_dx(_DT_CODE[x.dtype], dx.ptr, g.ptr, x.ptr, M, C, mr.ptr, gamma.ptr,
                      sums.ptr if sums is not None else None):
        _raise("tnn_bn_dx")
    return dx


# Pointwise losses (csrc/loss.cu): MSE, MAE, Huber, sigmoid cross-entropy; the kind codes of
# include/tnn_b200.h
LOSS_MSE, LOSS_MAE, LOSS_HUBER, LOSS_SIGMOID_CE = range(4)


def pointwise_loss(p, t, kind, m_global, delta=1.0, want_dp=False):
    """(loss, dp): L = (1/m_global) sum l(p, t) over every element, one launch; with want_dp the same
    pass also writes dL/dp for the upstream gradient 1 (else dp is None): what pointwise_loss_bwd
    computes from backward()'s default seed, bit for bit"""
    loss = empty((), p.dtype)
    dp = empty(p.shape, p.dtype) if want_dp else None
    if _lib.tnn_pointwise_loss(_DT_CODE[p.dtype], int(kind), p.ptr, t.ptr, p.size, float(m_global),
                               float(delta), loss.ptr, dp.ptr if want_dp else None):
        _raise("tnn_pointwise_loss")
    return loss, dp


def pointwise_loss_bwd(p, t, kind, m_global, delta, g):
    """dL/dp for the upstream gradient g (a scalar device array)"""
    dp = empty(p.shape, p.dtype)
    if g.dtype != p.dtype:
        g = astype(g, p.dtype)
    if _lib.tnn_pointwise_loss_bwd(_DT_CODE[p.dtype], int(kind), dp.ptr, p.ptr, t.ptr, p.size, float(m_global),
                                   float(delta), g.ptr):
        _raise("tnn_pointwise_loss_bwd")
    return dp


def ce_stats(z):
    B, C = z.shape
    stats = empty((2,), z.dtype)
    if _lib.tnn_ce_stats(_DT_CODE[z.dtype], z.ptr, B, C, stats.ptr):
        _raise("tnn_ce_stats")
    return stats


def ce_merge_stats(stats_all, n_ranks):
    out = empty((2,), stats_all.dtype)
    if _lib.tnn_ce_merge_stats(_DT_CODE[stats_all.dtype], out.ptr, stats_all.ptr, n_ranks):
        _raise("tnn_ce_merge_stats")
    return out


def _ce_labels(y):
    """(dense pointer, class-index pointer): a one-hot matrix that exists only as indices is passed as
    indices"""
    if type(y) is LazyOneHot and y._real is None:
        return None, y.labels_ptr
    return y.ptr, None


def ce_loss(z, y, stats, m_global):
    B, C = z.shape
    q = empty((B,), z.dtype)
    loss = empty((), z.dtype)
    y_ptr, lab_ptr = _ce_labels(y)
    if _lib.tnn_ce_loss(_DT_CODE[z.dtype], z.ptr, _DT_CODE[y.dtype], y_ptr, B, C, stats.ptr,
                        float(m_global), q.ptr, loss.ptr, lab_ptr):
        _raise("tnn_ce_loss")
    return loss, q


def ce_small_ok(B, C):
    return B <= 2048 and B * C <= 16384


def ce_fwd_small(z, y, m_global, want_dz=False):
    """stats, loss and q of a small logits matrix in one launch; with want_dz also dL/dz for the
    upstream gradient 1 (returned fourth, else None): what ce_bwd would compute from backward()'s
    default seed, bit for bit"""
    B, C = z.shape
    stats, q, loss = empty((2,), z.dtype), empty((B,), z.dtype), empty((), z.dtype)
    dz = empty((B, C), z.dtype) if want_dz else None
    if _lib.tnn_ce_fwd_small(_DT_CODE[z.dtype], z.ptr, _DT_CODE[y.dtype], y.ptr, B, C,
                             float(m_global), stats.ptr, q.ptr, loss.ptr, dz.ptr if want_dz else None):
        _raise("tnn_ce_fwd_small")
    return stats, loss, q, dz


def is_ones_scalar(g):
    """is this the shared constant backward() seeds a scalar loss with"""
    one = _ONES.get(np.dtype(g.dtype))
    return one is not None and g is one


def ce_bwd(z, y, stats, q, m_global, g):
    B, C = z.shape
    dz = empty((B, C), z.dtype)
    if g.dtype != z.dtype:
        g = astype(g, z.dtype)
    # a gradient this large feeds tensor-core products: the kernel also records max|dz| for their split
    stat = None
    if z.dtype == F32 and TC_SPLIT == "f16" and TC_ENABLED and B * C >= (1 << 16):
        stat = _new_meta()
        if _lib.tnn_f16_meta_reset(stat.ptr):
            _raise("tnn_f16_meta_reset")
    y_ptr, lab_ptr = _ce_labels(y)
    if _lib.tnn_ce_bwd(_DT_CODE[z.dtype], dz.ptr, z.ptr, _DT_CODE[y.dtype], y_ptr, B, C, stats.ptr,
                       q.ptr, float(m_global), g.ptr, stat.ptr if stat is not None else None, lab_ptr):
        _raise("tnn_ce_bwd")
    if stat is not None:
        dz.split = {"epoch": _split_epoch, "stat": stat}
    return dz


class MLPTail(object):
    """Workspace and argument block of the fused small-MLP tail pass (tnn_mlp_tail_step) for one
    network / batch size: layers 2..L of a Dense/ReLU MLP whose tail weights fit in shared memory."""

    MAX_WIDTH = 256
    MAX_LAYERS = 6
    SMEM_LIMIT = 220 * 1024

    def __init__(self, dims, batch, n_grad):
        """dims = [in0, out0 = in1, ..., out_{L-1}] of the tail layers; n_grad = length of the
        tail's stretch of the flat gradient arena (slot padding included)"""
        L = len(dims) - 1
        self.L, self.batch, self.n_grad = L, batch, n_grad
        self.in_dims = (_c_i64 * L)(*dims[:-1])
        self.out_dims = (_c_i64 * L)(*dims[1:])
        smem, n_ctas, scratch = _c_i64(), _c_i64(), _c_i64()
        if _lib.tnn_mlp_tail_workspace(L, self.in_dims, self.out_dims, batch, ctypes.byref(smem),
                                       ctypes.byref(n_ctas), ctypes.byref(scratch)):
            _raise("tnn_mlp_tail_workspace")
        self.smem_bytes, self.n_ctas = smem.value, n_ctas.value
        self.scratch = empty((scratch.value,), F32)   # layer inputs and dL/dz rows between the two phases
        self.stats = zeros((2 * self.n_ctas,), F32)
        self.loss_part = zeros((self.n_ctas,), F32)
        self.counters = zeros((16,), F32)             # uint32 rendezvous counters, rearmed by the kernel
        self.logits = empty((batch, dims[-1]), F32)   # the network's output rows of the last pass
        # dL/dlogits of the last pass: the last layer's dL/dz rows in the phase-1 -> phase-2 scratch
        self.dlogits = self.scratch.view((batch, dims[-1]), scratch.value - batch * dims[-1])

    @classmethod
    def eligible(cls, dims, batch):
        init()
        L = len(dims) - 1
        if not (1 <= L <= cls.MAX_LAYERS) or any(d < 1 or d > cls.MAX_WIDTH for d in dims):
            return False
        if batch < 1 or batch > 256:
            return False
        floats = sum(dims[i] * (dims[i + 1] | 1) + (dims[i + 1] + 3) // 4 * 4 for i in range(L))
        floats = (floats + 3) // 4 * 4 + 12 * sum(dims) + 4 * 256
        return floats * 4 <= cls.SMEM_LIMIT

    def run(self, ws, bs, grad_base, grad_offsets, n_grad, z1, y, m_global, dz1, loss_out):
        """ws/bs: device arrays of the tail parameters; grad_base: DArray view at the first tail
        parameter's gradient slot; grad_offsets: [dW_0, db_0, dW_1, ...] element offsets from it"""
        if n_grad != self.n_grad:
            raise ValueError("MLPTail was laid out for %d gradient elements, got %d" % (self.n_grad, n_grad))
        wp = (_c_vp * self.L)(*[w.ptr for w in ws])
        bp = (_c_vp * self.L)(*[b.ptr for b in bs])
        go = (_c_i64 * (2 * self.L))(*grad_offsets)
        if _lib.tnn_mlp_tail_step(self.L, self.in_dims, self.out_dims, wp, bp, go, grad_base.ptr, n_grad,
                                  z1.ptr, y.ptr, _DT_CODE[y.dtype], self.batch, float(m_global), dz1.ptr,
                                  loss_out.ptr, self.scratch.ptr, self.stats.ptr, self.loss_part.ptr,
                                  self.counters.ptr, self.logits.ptr):
            _raise("tnn_mlp_tail_step")


def opt_step(opt, param, step_out, grad, s0, s1, hyper):
    n = grad.size
    if isinstance(hyper, DArray):    # captured step: coefficients live in device memory
        if _lib.tnn_opt_step_dev(opt, _DT_CODE[grad.dtype], param.ptr if param is not None else None,
                                 step_out.ptr if step_out is not None else None, grad.ptr,
                                 s0.ptr if s0 is not None else None,
                                 s1.ptr if s1 is not None else None, n, hyper.ptr):
            _raise("tnn_opt_step_dev")
        return
    h = (_c_dbl * len(hyper))(*hyper)
    if _lib.tnn_opt_step(opt, _DT_CODE[grad.dtype], param.ptr if param is not None else None,
                         step_out.ptr if step_out is not None else None, grad.ptr,
                         s0.ptr if s0 is not None else None, s1.ptr if s1 is not None else None,
                         n, h, len(hyper)):
        _raise("tnn_opt_step")


# --------------------------------------------------------------------------------------------
# pinned host staging + copy stream (input prefetch), events, profiling
# --------------------------------------------------------------------------------------------
class PinnedArray(object):
    """numpy array backed by cudaHostAlloc memory"""

    def __init__(self, shape, dtype):
        init()
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)
        nbytes = max(_prod(self.shape), 1) * self.dtype.itemsize
        p = _c_vp()
        if _lib.tnn_host_alloc(nbytes, ctypes.byref(p)):
            _raise("tnn_host_alloc")
        self.ptr = p.value
        self.nbytes = nbytes
        raw = (ctypes.c_char * nbytes).from_address(self.ptr)
        self.array = np.frombuffer(raw, dtype=self.dtype, count=_prod(self.shape)).reshape(self.shape)

    def __del__(self):
        try:
            if self.ptr and _lib is not None:
                self.array = None
                _lib.tnn_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


class RegisteredHostArray(object):
    """a caller-owned C-contiguous numpy array pinned in place (cudaHostRegister) for the lifetime
    of this object"""

    def __init__(self, array):
        init()
        if not (isinstance(array, np.ndarray) and array.flags["C_CONTIGUOUS"]):
            raise ValueError("only C-contiguous numpy arrays can be pinned in place")
        self.array = array
        self.ptr = array.ctypes.data
        if _lib.tnn_host_register(self.ptr, array.nbytes):
            _raise("tnn_host_register")

    def row_address(self, row):
        return self.ptr + row * self.array.strides[0]

    def __del__(self):
        try:
            if self.ptr and _lib is not None:
                _lib.tnn_host_unregister(self.ptr)
                self.ptr = None
        except Exception:
            pass


def h2d_prefetch(dst, pinned):
    """queue pinned -> dst on the copy stream, after everything queued so far on compute.
    `pinned` is a PinnedArray / RegisteredHostArray or a raw address inside pinned memory."""
    if _lib.tnn_copy_wait_compute():
        _raise("tnn_copy_wait_compute")
    src = pinned if isinstance(pinned, int) else pinned.ptr
    if _lib.tnn_h2d_async_copy_stream(dst.ptr, src, dst.nbytes):
        _raise("tnn_h2d_async_copy_stream")


def copy_stream_sync():
    """host waits for the copy stream: a pinned staging buffer may be rewritten afterwards"""
    if _lib.tnn_copy_stream_sync():
        _raise("tnn_copy_stream_sync")


def wait_prefetch():
    if _lib.tnn_compute_wait_copy():
        _raise("tnn_compute_wait_copy")


_pinned_free = {}    # nbytes -> [PinnedArray]: read-back staging buffers are recycled


class AsyncRead(object):
    """Read-back of a device array that does not drain the compute stream: the copy runs on its own
    stream after the work queued so far; result() waits for it only (later steps stay queued)."""

    def __init__(self, d):
        init()
        self.shape, self.dtype = d.shape, d.dtype
        nbytes = max(d.nbytes, 1)
        free = _pinned_free.get(nbytes)
        self.pin = free.pop() if free else PinnedArray((nbytes,), np.uint8)
        self.event = Event()
        self._src = d                      # keeps the block alive until the copy has run
        self._value = None
        if _lib.tnn_d2h_async(self.pin.ptr, d.ptr, d.nbytes, self.event.ptr):
            _raise("tnn_d2h_async")

    def result(self):
        if self._value is None:
            if _lib.tnn_event_sync(self.event.ptr):
                _raise("tnn_event_sync")
            n = int(np.prod(self.shape)) if self.shape else 1
            self._value = np.frombuffer(self.pin.array, dtype=self.dtype, count=n).reshape(self.shape).copy()
            _pinned_free.setdefault(self.pin.nbytes, []).append(self.pin)
            self.pin = self._src = None
        return self._value


class Event(object):
    def __init__(self):
        init()
        p = _c_vp()
        if _lib.tnn_event_create(ctypes.byref(p)):
            _raise("tnn_event_create")
        self.ptr = p.value

    def record(self):
        if _lib.tnn_event_record(self.ptr):
            _raise("tnn_event_record")

    def elapsed_ms_since(self, start):
        ms = ctypes.c_float()
        if _lib.tnn_event_elapsed_ms(start.ptr, self.ptr, ctypes.byref(ms)):
            _raise("tnn_event_elapsed_ms")
        return ms.value

    def __del__(self):
        try:
            if self.ptr and _lib is not None:
                _lib.tnn_event_destroy(self.ptr)
        except Exception:
            pass


_LIVE_GRAPHS = weakref.WeakSet()


def destroy_all_graphs():
    """Recorded steps that contain NCCL collectives keep the communicator referenced: they have to
    go before the communicator does (core._dist.destroy_process_group calls this)."""
    for g in list(_LIVE_GRAPHS):
        g.destroy()


class StepGraph(object):
    """A recorded sequence of device work (CUDA graph) that replay() re-issues with one call.

        g = StepGraph()
        with g.capture():
            ... any device ops: they are recorded, not executed ...
        g.replay()

    Blocks allocated inside capture() belong to the graph until it is destroyed."""

    def __init__(self):
        init()
        self.handle = None
        _LIVE_GRAPHS.add(self)

    def capture(self):
        return _Capture(self)

    def replay(self):
        if not self.handle:
            raise BackendError("this recorded step was destroyed (process group torn down?)")
        if _lib.tnn_graph_launch(self.handle):
            _raise("tnn_graph_launch")

    def info(self):
        a, b, c = _c_sz(), _c_sz(), _c_sz()
        if _lib.tnn_graph_info(self.handle, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)):
            _raise("tnn_graph_info")
        return {"nodes": a.value, "kernel_nodes": b.value, "blocks": c.value}

    def destroy(self):
        if self.handle and _lib is not None:
            _lib.tnn_graph_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class _Capture(object):
    def __init__(self, graph):
        self.graph = graph

    def __enter__(self):
        if self.graph.handle:
            raise BackendError("StepGraph already holds a captured step")
        # the cyclic garbage collector must not run finalisers (which may synchronise the stream or
        # free pinned memory) in the middle of a capture: collect now, pause it until the end
        global _capturing
        gc.collect()
        self._gc_was_enabled = gc.isenabled()
        gc.disable()
        if _lib.tnn_graph_begin():
            if self._gc_was_enabled:
                gc.enable()
            _raise("tnn_graph_begin")
        _capturing = True
        return self.graph

    def __exit__(self, exc_type, exc, tb):
        global _capturing
        _capturing = False
        try:
            if exc_type is not None:
                _lib.tnn_graph_abort()
                return False
            h = _c_vp()
            if _lib.tnn_graph_end(ctypes.byref(h)):
                _raise("tnn_graph_end")
            self.graph.handle = h.value
            return False
        finally:
            if self._gc_was_enabled:
                gc.enable()


def prof_enable(family):
    init()
    if _lib.tnn_prof_enable(family):
        _raise("tnn_prof_enable")


def prof_collect():
    ms, n = _c_dbl(), ctypes.c_uint64()
    if _lib.tnn_prof_collect(ctypes.byref(ms), ctypes.byref(n)):
        _raise("tnn_prof_collect")
    return ms.value, n.value


def l2_flush():
    init()
    if _lib.tnn_l2_flush():
        _raise("tnn_l2_flush")
