"""ctypes binding of libb200agg.so (include/b200agg.h).

This is the reference-side binding a vaex maintainer would add: vaex loads its native kernels as the pybind11
modules ``vaex.superagg`` / ``vaex.superutils`` (packages/vaex-core/src/agg.cpp:91, src/superutils.cpp:214);
here the same entry points are reached through a plain C ABI.  There is NO CPU fallback: if the shared library or a
usable sm_100 device is missing every compute call raises.
"""
import ctypes as C
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# VAEX_B200_LIB: load this build of the library instead of the in-tree one (A/B timing of kernel variants on one box)
LIB_PATH = os.environ.get("VAEX_B200_LIB") or os.path.join(_HERE, "libb200agg.so")
CSRC = os.path.join(_HERE, "csrc")
SOURCES = ["api.cu", "binby.cu", "expr.cu", "fast.cu", "first.cu", "hashset.cu", "list.cu", "minmax.cu", "nunique.cu", "ringcount.cu", "tilesort.cu"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]

DTYPES = ["float64", "float32", "int64", "int32", "int16", "int8", "uint64", "uint32", "uint16", "uint8", "bool"]
DTYPE_CODE = {n: i for i, n in enumerate(DTYPES)}
F64, F32, I64, I32, I16, I8, U64, U32, U16, U8, BOOL = range(11)
BINNER_SCALAR, BINNER_ORDINAL, BINNER_HASH = 0, 1, 2
AGG_COUNT, AGG_SUM, AGG_SUM_MOMENT, AGG_MIN, AGG_MAX, AGG_FIRST, AGG_LAST, AGG_NUNIQUE, AGG_LIST, AGG_LIST_STRING = range(10)
MEM_HOST, MEM_DEVICE, MEM_MIXED = 0, 1, 2
FLAG_ASYNC_HOST = 1
ERR_NODATA = -3


class Binner(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dtype", C.c_int32), ("byteswap", C.c_int32), ("allow_other", C.c_int32), ("invert", C.c_int32),
                ("reserved", C.c_int32), ("vmin", C.c_double), ("vmax", C.c_double), ("bins", C.c_uint64), ("ordinal_count", C.c_int64),
                ("min_value", C.c_int64), ("set", C.c_void_p), ("data", C.c_void_p), ("mask", C.c_void_p)]


class ExprOp(C.Structure):
    _fields_ = [("op", C.c_int32), ("cls", C.c_int32), ("arg", C.c_int32), ("reserved", C.c_int32), ("f", C.c_double), ("i", C.c_int64)]


class ExprInput(C.Structure):
    _fields_ = [("data", C.c_void_p), ("dtype", C.c_int32), ("reserved", C.c_int32)]


class AggInput(C.Structure):
    _fields_ = [("agg", C.c_void_p), ("data", C.c_void_p), ("order", C.c_void_p), ("mask", C.c_void_p)]


def build(force=False, verbose=False):
    """Compile libb200agg.so for sm_100a in-tree (nvcc cross-compiles without a GPU): one object per source (only stale ones are
    rebuilt, in parallel), then one link."""
    from concurrent.futures import ThreadPoolExecutor
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")] + [os.path.join(_HERE, "..", "include", "b200agg.h")]
    hdr_time = max(os.path.getmtime(h) for h in hdrs)
    objdir = os.path.join(CSRC, "_obj")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    jobs, objs = [], []
    for src in SOURCES:
        path, obj = os.path.join(CSRC, src), os.path.join(objdir, src[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(path), hdr_time):
            jobs.append(["nvcc"] + flags + ["-c", "-o", obj, path])
    if not jobs and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(o) for o in objs):
        return LIB_PATH

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs)
    return LIB_PATH


_lib = None
_lock = threading.RLock()


def lib():
    """The loaded library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(vaex_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        i32, i64, u32, u64, vp, sz = C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_void_p, C.c_size_t
        P = C.POINTER
        sig = {
            "b200_last_error": (C.c_char_p, []),
            "b200_abi_version": (i32, []),
            "b200_device_count": (i32, []),
            "b200_ctx_create": (i32, [i32, i32, P(vp)]),
            "b200_ctx_destroy": (i32, [vp]),
            "b200_ctx_sync": (i32, [vp, i32]),
            "b200_ctx_device": (i32, [vp]),
            "b200_ctx_stream": (i32, [vp, i32, P(vp)]),
            "b200_ctx_path_stats": (i32, [vp, i32, P(u64)]),
            "b200_ctx_host_stats": (i32, [vp, P(u64), i32]),
            "b200_ctx_occupy": (i32, [vp, i32, i32, i32, i32, u64]),
            "b200_agg_create": (i32, [vp, i32, i32, i32, i32, u32, u64, P(vp)]),
            "b200_agg_destroy": (i32, [vp]),
            "b200_agg_reset": (i32, [vp]),
            "b200_agg_reset_on": (i32, [vp, i32]),
            "b200_agg_read_on": (i32, [vp, i32, vp]),
            "b200_agg_cells": (u64, [vp]),
            "b200_agg_result_dtype": (i32, [vp]),
            "b200_agg_bytes": (sz, [vp]),
            "b200_agg_device_ptr": (i32, [vp, i32, P(vp), P(sz)]),
            "b200_agg_device_dtype": (i32, [vp]),
            "b200_agg_read": (i32, [vp, vp, vp]),
            "b200_agg_merge": (i32, [vp, P(vp), i32]),
            "b200_agg_list_finish": (i32, [vp, P(i64)]),
            "b200_agg_list_read": (i32, [vp, vp, vp]),
            "b200_agg_list_string_finish": (i32, [vp, P(i64), P(i64)]),
            "b200_agg_list_string_read": (i32, [vp, vp, vp, vp, vp]),
            "b200_agg_write": (i32, [vp, vp]),
            "b200_bin": (i32, [vp, i32, P(Binner), i32, P(AggInput), i32, i64, i64, i32, u32]),
            "b200_eval": (i32, [vp, i32, P(ExprOp), i32, P(ExprInput), i32, P(vp), i32, i64, i32, i32, vp]),
            "b200_compact": (i32, [vp, i32, vp, i32, P(vp), P(i32), i64, i32, P(vp), P(i64)]),
            "b200_set_dtype": (i32, [vp]),
            "b200_strset_create": (i32, [vp, i32, i64, P(vp)]),
            "b200_strset_update": (i32, [vp, i32, vp, vp, vp, i64, i32, vp, vp, i32]),
            "b200_strset_map_ordinal": (i32, [vp, i32, vp, vp, vp, i64, vp, i32, i32]),
            "b200_strset_key_bytes": (i32, [vp, P(i64)]),
            "b200_strset_key_array": (i32, [vp, vp, vp]),
            "b200_set_create": (i32, [vp, i32, i32, i64, P(vp)]),
            "b200_set_from_keys": (i32, [vp, i32, vp, i64, i64, i64, i64, P(vp)]),
            "b200_set_destroy": (i32, [vp]),
            "b200_set_update": (i32, [vp, i32, vp, vp, i64, i64, i32, vp, vp, i32, u32]),
            "b200_set_merge": (i32, [vp, P(vp), i32]),
            "b200_set_count": (i64, [vp]),
            "b200_set_nan_count": (i64, [vp]),
            "b200_set_null_count": (i64, [vp]),
            "b200_set_nan_index": (i64, [vp]),
            "b200_set_null_index": (i64, [vp]),
            "b200_set_nmaps": (i32, [vp]),
            "b200_set_offsets": (i32, [vp, vp]),
            "b200_set_key_array": (i32, [vp, vp]),
            "b200_set_ordinal_dtype": (i32, [vp]),
            "b200_set_map_ordinal": (i32, [vp, i32, vp, i64, vp, i32, u32]),
            "b200_set_isin": (i32, [vp, i32, vp, i64, vp, i32, u32]),
            "b200_set_combine": (i32, [vp, i32, i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), i64, vp, i32, u32]),
            "b200_set_bytes": (sz, [vp]),
            "b200_counter_create": (i32, [vp, i32, i32, P(vp)]),
            "b200_set_counts": (i32, [vp, vp]),
            "b200_minmax": (i32, [vp, i32, i32, i32, vp, vp, i64, i32, vp]),
            "b200_host_register": (i32, [vp, sz]),
            "b200_host_unregister": (i32, [vp]),
            "b200_hash64": (u64, [u64]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        if L.b200_abi_version() != 1:
            raise RuntimeError("libb200agg.so ABI version mismatch")
        _lib = L
    return _lib


EXPORTED_SYMBOLS = None  # filled by tests from include/b200agg.h


def check(rc):
    if rc == 0:
        return
    msg = lib().b200_last_error().decode()
    if rc == -6:
        raise MemoryError(msg)
    raise RuntimeError(msg)


# ------------------------------------------------------------------------------------------------
# contexts: one per (device); slots play the role of the reference's thread index
# ------------------------------------------------------------------------------------------------
class Context:
    def __init__(self, device=None, nslots=64):
        if device is None:
            device = default_device()
        h = C.c_void_p()
        check(lib().b200_ctx_create(int(device), int(nslots), C.byref(h)))
        self._h = h
        self.device = int(device)
        self.nslots = int(nslots)

    def slot(self, thread):
        return int(thread) % self.nslots

    def sync(self, slot=-1):
        check(lib().b200_ctx_sync(self._h, int(slot)))

    def path_stats(self, slot=0):
        """Counters of the last partitioned count(*) batch on this slot (include/b200agg.h b200_ctx_path_stats)."""
        out = (C.c_uint64 * 6)()
        check(lib().b200_ctx_path_stats(self._h, int(slot), out))
        return dict(rows=out[0], entries=out[1], chunks=out[2], chunk_entries=out[3], memset_bytes=out[4], lists=out[5])

    def host_stats(self, reset=False):
        """Where the host-chunk path spent its wall time (include/b200agg.h b200_ctx_host_stats), milliseconds summed over slots."""
        out = (C.c_uint64 * 6)()
        check(lib().b200_ctx_host_stats(self._h, out, int(bool(reset))))
        return dict(wait_ms=out[0] / 1e6, memcpy_ms=out[1] / 1e6, enqueue_ms=out[2] / 1e6, bin_ms=out[3] / 1e6, pieces=out[4], calls=out[5])

    def stream(self, slot=0):
        s = C.c_void_p()
        check(lib().b200_ctx_stream(self._h, int(slot), C.byref(s)))
        return s.value or 0

    def close(self):
        if self._h:
            lib().b200_ctx_destroy(self._h)
            self._h = None


_contexts = {}


def default_device():
    env = os.environ.get("VAEX_B200_DEVICE")
    if env is not None:
        return int(env)
    import sys
    torch = sys.modules.get("torch")
    if torch is not None and torch.cuda.is_available():
        return torch.cuda.current_device()
    return int(os.environ.get("LOCAL_RANK", "0"))


def context(device=None):
    """Process-wide context of a device (created on first use)."""
    if device is None:
        device = default_device()
    with _lock:
        ctx = _contexts.get(device)
        if ctx is None:
            ctx = _contexts[device] = Context(device)
        return ctx


# ------------------------------------------------------------------------------------------------
# column marshalling: numpy arrays are host buffers, anything with __cuda_array_interface__ is device memory
# ------------------------------------------------------------------------------------------------
class Column:
    __slots__ = ("ptr", "memspace", "dtype", "code", "byteswap", "length", "keep")


def _np_dtype_code(dt):
    dt = np.dtype(dt)
    if dt.kind in "mM":
        return DTYPE_CODE["int64"] if dt.kind == "m" else DTYPE_CODE["uint64"]
    name = dt.newbyteorder("=").name
    if name not in DTYPE_CODE:
        raise RuntimeError(f"dtype {dt} is not supported by the binned-statistics kernels")
    return DTYPE_CODE[name]


def column(ar, expected_itemsize=None):
    c = Column()
    cai = getattr(ar, "__cuda_array_interface__", None)
    if cai is not None and not isinstance(ar, np.ndarray):
        shape = cai["shape"]
        if len(shape) != 1:
            raise RuntimeError("Expected a 1d array")
        dt = np.dtype(cai["typestr"])
        strides = cai.get("strides")
        if strides is not None and shape[0] > 1 and strides[0] != dt.itemsize:
            raise RuntimeError("device columns must be contiguous")
        c.ptr = cai["data"][0]
        c.memspace = MEM_DEVICE
        c.dtype = dt
        c.length = shape[0]
        c.keep = ar
    else:
        a = np.asarray(ar)
        if a.ndim != 1:
            raise RuntimeError("Expected a 1d array")
        if a.dtype.kind in "mM":
            a = a.view("uint64")  # the reference passes datetimes as integers (vaex/cpu.py:692-694)
        if not a.flags.c_contiguous:
            a = np.ascontiguousarray(a)
        c.ptr = a.ctypes.data if a.size else 0
        c.memspace = MEM_HOST
        c.dtype = a.dtype
        c.length = a.shape[0]
        c.keep = a
    if expected_itemsize is not None and c.dtype.itemsize != expected_itemsize:
        raise RuntimeError("Itemsize of data and binner are not equal")
    c.code = _np_dtype_code(c.dtype)
    c.byteswap = int(c.dtype.byteorder not in ("=", "|") and c.dtype.byteorder != ("<" if np.little_endian else ">"))
    return c


def mask_column(ar):
    """uint8/bool mask -> Column (bool viewed as uint8)."""
    cai = getattr(ar, "__cuda_array_interface__", None)
    if cai is not None and not isinstance(ar, np.ndarray):
        c = column(ar)
        if c.dtype.itemsize != 1:
            raise RuntimeError("masks must be 1 byte per row")
        return c
    a = np.asarray(ar)
    if a.ndim != 1:
        raise RuntimeError("Expected a 1d array")
    if a.dtype == np.bool_:
        a = np.ascontiguousarray(a).view(np.uint8)
    elif a.dtype.itemsize != 1:
        a = a.astype(np.uint8)
    return column(a)


class pinned:
    """Context manager / handle that page-locks numpy columns for the lifetime of a computation (b200_host_register)."""

    def __init__(self, *arrays):
        self.arrays = [a for a in arrays if isinstance(a, np.ndarray) and a.size and a.flags.c_contiguous]
        context()  # cudaHostRegister needs a CUDA context
        for a in self.arrays:
            check(lib().b200_host_register(a.ctypes.data, a.nbytes))

    def release(self):
        for a in self.arrays:
            lib().b200_host_unregister(a.ctypes.data)
        self.arrays = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.release()
