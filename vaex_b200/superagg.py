"""Drop-in mirror of the reference's native module ``vaex.superagg`` on top of libb200agg.so.

Same class names (``Binner{Scalar,Ordinal}_<dtype>[_non_native]``, ``Grid``, ``Agg{Count,Sum,SumMoment,Min,Max}_<dtype>``,
``AggFirst_<dtype>_<dtype2>``), constructor arguments, methods and error messages as the pybind11 module built from
packages/vaex-core/src/agg.cpp:91-118, src/binners.cpp:92-146, src/binner_ordinal.cpp:212-251, src/agg_base.hpp:249-260, so
``vaex.utils.find_type_from_dtype(vaex_b200.superagg, "AggSum_", dtype)`` (vaex/utils.py:754-791) resolves exactly as it
does against the reference.  The per-row work happens in the CUDA kernels behind ``b200_bin``; buffers handed to
``set_data`` may be numpy arrays (staged host->device per call) or device arrays (anything exposing
``__cuda_array_interface__``, e.g. torch CUDA tensors; zero copy).

Differences, all deliberate:
  * ``grids`` is accepted but ONE device grid is kept (atomics replace the reference's per-thread copies, src/agg_base.hpp:33-77);
  * ``thread`` selects a CUDA stream + staging arena instead of a private pointer table.
"""
import ctypes as C
import sys
import types

import numpy as np

from . import _lib

_DT = _lib.DTYPES


class Binner:
    """Base class (the reference's ``vaex.superagg.Binner``, src/agg.hpp:32-41)."""

    def __init__(self, threads, expression):
        self.threads = int(threads)
        self.expression = expression
        self._data = {}
        self._mask = {}

    def set_data(self, thread, ar):
        self._data[int(thread)] = _lib.column(ar, self._itemsize)

    def set_data_mask(self, thread, ar):
        self._mask[int(thread)] = _lib.mask_column(ar)

    def clear_data_mask(self, thread):
        self._mask.pop(int(thread), None)

    def data_length(self, thread):
        return self._data[int(thread)].length

    def _fill(self, b, thread):
        raise NotImplementedError


class _BinnerScalar(Binner):
    _dtype = None
    _non_native = False

    def __init__(self, threads, expression, vmin, vmax, bins):
        super().__init__(threads, expression)
        self.vmin = float(vmin)
        self.vmax = float(vmax)
        self.bins = int(bins)

    def copy(self):
        return type(self)(self.threads, self.expression, self.vmin, self.vmax, self.bins)

    def __len__(self):
        return self.bins + 3  # src/binners.cpp:59

    def __reduce__(self):
        return type(self), (self.threads, self.expression, self.vmin, self.vmax, self.bins)

    def __repr__(self):
        return f"<{type(self).__name__} expression={self.expression!r} vmin={self.vmin} vmax={self.vmax} bins={self.bins}>"

    def _fill(self, b, thread):
        col = self._data.get(thread)
        if col is None:
            raise RuntimeError("data not set")
        b.kind = _lib.BINNER_SCALAR
        b.dtype = self._code
        b.byteswap = int(self._non_native)
        b.vmin, b.vmax, b.bins = self.vmin, self.vmax, self.bins
        b.data = col.ptr
        m = self._mask.get(thread)
        b.mask = m.ptr if m is not None else None
        return [col] + ([m] if m is not None else [])


class _BinnerOrdinal(Binner):
    _dtype = None
    _non_native = False

    def __init__(self, threads, expression, ordinal_count, min_value=0, allow_other=False, invert=False):
        super().__init__(threads, expression)
        self.ordinal_count = int(ordinal_count)
        self.min_value = int(min_value)
        self.allow_other = bool(allow_other)
        self.invert = bool(invert)

    def copy(self):
        return type(self)(self.threads, self.expression, self.ordinal_count, self.min_value, self.allow_other, self.invert)

    def __len__(self):
        return self.ordinal_count + (3 if self.allow_other else 2)  # src/binner_ordinal.cpp:178

    def __reduce__(self):
        return type(self), (self.threads, self.expression, self.ordinal_count, self.min_value, self.allow_other, self.invert)

    def __repr__(self):
        return f"<{type(self).__name__} expression={self.expression!r} count={self.ordinal_count} min={self.min_value}>"

    def _fill(self, b, thread):
        col = self._data.get(thread)
        if col is None:
            raise RuntimeError("data not set")
        b.kind = _lib.BINNER_ORDINAL
        b.dtype = self._code
        b.byteswap = int(self._non_native)
        b.ordinal_count, b.min_value = self.ordinal_count, self.min_value
        b.allow_other, b.invert = int(self.allow_other), int(self.invert)
        b.data = col.ptr
        m = self._mask.get(thread)
        b.mask = m.ptr if m is not None else None
        return [col] + ([m] if m is not None else [])


class _BinnerHash(Binner):
    """Ordinal binner fed by a fused device probe of an ordered_set (no materialised code column).

    Takes the place of the reference's ``_ordinal_values(key, set)`` virtual column + ``BinnerOrdinal``
    (vaex/groupby.py:303-317).  Unknown keys land in the null cell like ``-1`` codes do there
    (src/binner_ordinal.cpp:166-167); the reference's experimental ``BinnerHash`` (src/binner_hash.cpp, off by default and
    writing out of bounds for unknown keys) is NOT what this mirrors."""
    _dtype = None
    _non_native = False

    def __init__(self, threads, expression, hash_map, allow_other=False, invert=False):
        super().__init__(threads, expression)
        self.hash_map = getattr(hash_map, "_internal", hash_map)
        self.allow_other = bool(allow_other)
        self.invert = bool(invert)

    @property
    def ordinal_count(self):
        return len(self.hash_map)

    def copy(self):
        return type(self)(self.threads, self.expression, self.hash_map, self.allow_other, self.invert)

    def __len__(self):
        return self.ordinal_count + (3 if self.allow_other else 2)

    def _fill(self, b, thread):
        col = self._data.get(thread)
        if col is None:
            raise RuntimeError("data not set")
        b.kind = _lib.BINNER_HASH
        b.dtype = self._code
        b.ordinal_count, b.min_value = self.ordinal_count, 0
        b.allow_other, b.invert = int(self.allow_other), int(self.invert)
        b.set = self.hash_map._h
        b.data = col.ptr
        m = self._mask.get(thread)
        b.mask = m.ptr if m is not None else None
        return [col] + ([m] if m is not None else [])


class BinnerCombined:
    """``vaex.superagg.BinnerCombined(threads, binners)`` (src/binner_combined.cpp:5-36): a binner made of several binners whose
    indices are composed with strides 1, shape_0, shape_0 * shape_1, ... (``to_bins`` :25-29).  The reference binds it WITHOUT the
    Binner base class (:40-44), so its own ``Grid`` cannot take one; here a Grid simply flattens it into its members, which is what
    the composed strides amount to.  ``len()`` reports the LAST member's shape, like the reference's ``shape()`` (:31)."""

    def __init__(self, threads, binners):
        self.threads = int(threads)
        self.binners = list(binners)
        self.expression = ""
        self.shapes = [len(b) for b in self.binners]
        self.strides = []
        s = 1
        for n in self.shapes:
            self.strides.append(s)
            s *= n

    def copy(self):
        return BinnerCombined(self.threads, self.binners)

    def __len__(self):
        return self.shapes[-1]

    def data_length(self, thread):
        return self.binners[0].data_length(thread)

    def __reduce__(self):
        return (BinnerCombined, (self.threads, self.binners))


class Grid:
    """``vaex.superagg.Grid`` (src/agg.hpp:53-143): shapes/strides with the first binner fastest + the bin() driver."""

    def __init__(self, binners):
        flat = []
        for b in binners:  # a BinnerCombined contributes its member binners, strides composed as its to_bins does
            flat.extend(b.binners if isinstance(b, BinnerCombined) else [b])
        self.binners = flat
        if len(self.binners) > 8:
            raise RuntimeError("at most 8 binners are supported")
        self.shapes = [len(b) for b in self.binners]
        self.strides = []
        s = 1
        for n in self.shapes:
            self.strides.append(s)
            s *= n
        self.length1d = s
        self._ctx = None

    def __len__(self):
        return self.length1d

    @property
    def dimensions(self):
        return len(self.binners)

    def bin(self, thread, aggregators, length=None, row_offset=0, flags=0):
        thread = int(thread)
        if length is None:
            if not self.binners:
                raise RuntimeError("no binners set and no length given")
            length = self.binners[0].data_length(thread)
        if not aggregators:
            return
        ctx = aggregators[0]._ctx
        nb = len(self.binners)
        B = (_lib.Binner * max(nb, 1))()
        keep = []
        for i, b in enumerate(self.binners):
            keep += b._fill(B[i], thread)
        na = len(aggregators)
        A = (_lib.AggInput * na)()
        for k, agg in enumerate(aggregators):
            keep += agg._fill(A[k], thread)
        spaces = {c.memspace for c in keep}
        # host and device columns in one call (device-computed group codes next to host value columns): every pointer is
        # classified by the library
        memspace = _lib.MEM_MIXED if len(spaces) > 1 else (spaces.pop() if spaces else _lib.MEM_HOST)
        for c in keep:
            if c.length < length:
                raise RuntimeError(f"a column of length {c.length} is shorter than the {length} rows to bin")
        _lib.check(_lib.lib().b200_bin(ctx._h, ctx.slot(thread), B, nb, A, na, int(length), int(row_offset), memspace, int(flags)))


class Aggregator:
    """``vaex.superagg.Aggregator`` (src/agg.hpp:43-51) over ONE device grid."""
    _op = None
    _dtype = None
    _dtype2 = "int64"
    _non_native = False

    def __init__(self, grid, grids, threads, *extra):
        self.grid = grid
        self.grids = int(grids)
        self.threads = int(threads)
        self._ctx = _lib.context()
        self._data = {}
        self._order = {}
        self._mask = {}
        self._extra = extra
        op, moment = self._op, 0
        if op == _lib.AGG_SUM_MOMENT:
            moment = int(extra[0])
        if op == _lib.AGG_FIRST and extra and extra[0]:
            op = _lib.AGG_LAST
        if op in (_lib.AGG_NUNIQUE, _lib.AGG_LIST, _lib.AGG_LIST_STRING):  # (dropmissing, dropnan) (src/agg_nunique.cpp:14) / (dropnan, dropnull) (src/agg_list.cpp:16)
            moment = int(bool(extra[0])) | (int(bool(extra[1])) << 1)
        self._h = C.c_void_p()
        _lib.check(_lib.lib().b200_agg_create(self._ctx._h, op, self._code, _lib.DTYPE_CODE[self._dtype2], int(self._non_native), moment, len(grid),
                                              C.byref(self._h)))
        self._result_dtype = np.dtype(_DT[_lib.lib().b200_agg_result_dtype(self._h)])

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                _lib.lib().b200_agg_destroy(h)
            except Exception:
                pass
            self._h = None

    # -- reference protocol --------------------------------------------------------------------------
    def set_data(self, thread, ar, index=0):
        col = _lib.column(ar)
        want = self._dtype2 if index == 1 else self._dtype
        if np.dtype(col.dtype).itemsize != np.dtype(want).itemsize:
            raise RuntimeError("Itemsize of data and aggregator are not equal")
        (self._order if index == 1 else self._data)[int(thread)] = col

    def set_data_mask(self, thread, ar):
        self._mask[int(thread)] = _lib.mask_column(ar)

    def clear_data_mask(self, thread):
        self._mask.pop(int(thread), None)

    def merge(self, others):
        if not others:
            return
        arr = (C.c_void_p * len(others))(*[o._h for o in others])
        _lib.check(_lib.lib().b200_agg_merge(self._h, arr, len(others)))

    def __sizeof__(self):
        # the reference reports sizeof(grid_type) * grids * cells (src/agg_base.hpp:34-35) and vaex asserts it equals its own
        # prediction (vaex/agg.py:311-318); report the same figure.  The bytes really held on the device: .device_bytes
        return int(_lib.lib().b200_agg_bytes(self._h)) * self.grids

    @property
    def device_bytes(self):
        return int(_lib.lib().b200_agg_bytes(self._h))

    def _read(self):
        n = len(self.grid)
        out = np.empty(n, self._result_dtype)
        mask = np.empty(n, np.uint8) if self._op == _lib.AGG_FIRST else None
        _lib.check(_lib.lib().b200_agg_read(self._h, out.ctypes.data, None if mask is None else mask.ctypes.data))
        return out, mask

    def get_result(self):
        out, mask = self._read()
        shapes = self.grid.shapes
        res = out.reshape(shapes, order="F")
        if mask is not None:  # numpy.ma like src/agg_first.cpp:100-113
            return np.ma.array(res, mask=mask.astype(bool).reshape(shapes, order="F"))
        return res

    def __array__(self, dtype=None, copy=None):
        # buffer protocol of the reference: shape (grids, *shapes) (src/agg_base.hpp:106-125); grid 0 carries everything
        out, _ = self._read()
        full = np.empty((self.grids,) + tuple(self.grid.shapes), self._result_dtype, order="F")
        fill = out.copy()
        self._identity(fill)
        for g in range(self.grids):
            full[g] = (out if g == 0 else fill).reshape(self.grid.shapes, order="F")
        return full if dtype is None else full.astype(dtype)

    def _identity(self, ar):
        if self._op == _lib.AGG_MIN or self._op == _lib.AGG_MAX:
            mx = self._op == _lib.AGG_MAX
            if ar.dtype.kind == "f":
                ar[:] = -np.inf if mx else np.inf
            elif ar.dtype.kind == "b":
                ar[:] = not mx
            else:
                info = np.iinfo(ar.dtype)
                ar[:] = info.min if mx else info.max
        else:
            ar[:] = 0

    def load(self, values):
        """TaskPartAggregation initial_values (vaex/cpu.py:654-658): values has the (grids, *shapes) buffer shape or one grid."""
        values = np.asarray(values)
        if values.ndim == len(self.grid.shapes) + 1:
            folded = self._fold(values)
        else:
            folded = values
        flat = np.ascontiguousarray(folded.reshape(-1, order="F"), dtype=self._result_dtype)
        _lib.check(_lib.lib().b200_agg_write(self._h, flat.ctypes.data))

    def _fold(self, values):
        if self._op == _lib.AGG_MIN:
            return values.min(axis=0)
        if self._op == _lib.AGG_MAX:
            return values.max(axis=0)
        return values.sum(axis=0, dtype=self._result_dtype)

    def reset(self, thread=None):
        """initial_fill() again; with `thread` the reset is only enqueued on that slot's stream (no host sync)."""
        if thread is None:
            _lib.check(_lib.lib().b200_agg_reset(self._h))
        else:
            _lib.check(_lib.lib().b200_agg_reset_on(self._h, self._ctx.slot(thread)))

    def read_async(self, thread, out):
        """Enqueue a D2H copy of the device grid (device cell dtype) into `out` (pinned host ndarray / tensor data_ptr)."""
        ptr = out.ctypes.data if isinstance(out, np.ndarray) else out.data_ptr()
        _lib.check(_lib.lib().b200_agg_read_on(self._h, self._ctx.slot(thread), ptr))

    def device_pointer(self, which=0):
        p = C.c_void_p()
        n = C.c_size_t()
        _lib.check(_lib.lib().b200_agg_device_ptr(self._h, which, C.byref(p), C.byref(n)))
        return p.value, n.value

    @property
    def device_dtype(self):
        return np.dtype(_DT[_lib.lib().b200_agg_device_dtype(self._h)])

    def _fill(self, a, thread):
        a.agg = self._h
        keep = []
        col = self._data.get(thread)
        if col is not None:
            a.data = col.ptr
            keep.append(col)
        elif self._op != _lib.AGG_COUNT:
            raise RuntimeError("data not set")
        o = self._order.get(thread)
        if o is not None:
            a.order = o.ptr
            keep.append(o)
        m = self._mask.get(thread)
        if m is not None:
            a.mask = m.ptr
            keep.append(m)
        return keep


class _AggNUnique(Aggregator):
    """``AggNUnique_<dtype>(grid, grids, threads, dropmissing, dropnan)`` (src/agg_nunique.cpp:7-92, bound at :200-211): number of
    distinct values per cell.  ``set_data_mask``: 0 = the row is null; ``set_selection_mask``: 0 = the row is skipped."""
    _op = _lib.AGG_NUNIQUE

    def __init__(self, grid, grids, threads, dropmissing, dropnan):
        self._selection = {}
        super().__init__(grid, grids, threads, dropmissing, dropnan)

    def set_selection_mask(self, thread, ar):
        self._selection[int(thread)] = _lib.mask_column(ar)

    def clear_selection_mask(self, thread):
        self._selection.pop(int(thread), None)

    def get_result(self):
        if self.grids != 1:
            raise RuntimeError("Expected 1 grid")  # src/agg_nunique.cpp:20-22
        return super().get_result()

    def merge(self, others):
        if others:
            raise RuntimeError("merge not implemented")  # src/agg_nunique.cpp:43-46

    def _fill(self, a, thread):
        keep = super()._fill(a, thread)
        s = self._selection.get(thread)
        if s is not None:
            a.order = s.ptr  # the C ABI carries the selection mask of NUNIQUE in the `order` slot (include/b200agg.h)
            keep.append(s)
        return keep


class _AggList(Aggregator):
    """``AggList_<dtype>(grid, grids, threads, dropnan, dropnull)`` (src/agg_list.cpp:5-127, bound at :246-259): per cell the list of
    the rows' values.  ``get_result()`` returns what the reference hands to ``vaex.arrow.convert.list_from_arrays``: a pyarrow list
    array with one list per cell (cells in the grid's flat order, first binner fastest)."""
    _op = _lib.AGG_LIST

    def __init__(self, grid, grids, threads, dropnan=False, dropnull=False):
        if int(grids) != 1:
            raise RuntimeError("list aggregation only accepts 1 grid")  # src/agg_list.cpp:18-20
        super().__init__(grid, grids, threads, dropnan, dropnull)

    def result_arrays(self):
        """(int64 offsets[cells + 1], flat values)"""
        total = C.c_int64(0)
        _lib.check(_lib.lib().b200_agg_list_finish(self._h, C.byref(total)))
        offsets = np.zeros(len(self.grid) + 1, np.int64)
        values = np.zeros(max(total.value, 1), np.dtype(self._dtype))
        _lib.check(_lib.lib().b200_agg_list_read(self._h, offsets.ctypes.data, values.ctypes.data))
        return offsets, values[:total.value]

    def get_result(self):
        import pyarrow as pa
        offsets, values = self.result_arrays()
        return pa.LargeListArray.from_arrays(pa.array(offsets), pa.array(values))

    def merge(self, others):
        pass  # src/agg_list.cpp:46

    def __sizeof__(self):
        return 0  # "cannot predict memory usage" (vaex/agg.py:306-309)


# ---- string aggregators (src/agg_count.cpp:70-195 AggCount_string, src/agg_nunique_string.cpp AggNUnique_string) ----------------
def _make(name, base, **attrs):
    cls = type(name, (base,), attrs)
    cls.__module__ = __name__
    globals()[name] = cls
    return cls


_AGG_OPS = {"AggCount": _lib.AGG_COUNT, "AggSum": _lib.AGG_SUM, "AggSumMoment": _lib.AGG_SUM_MOMENT, "AggMin": _lib.AGG_MIN, "AggMax": _lib.AGG_MAX}

for _name in _DT:
    for _nn in (False, True):
        _sfx = _name + ("_non_native" if _nn else "")
        _isz = np.dtype(_name).itemsize
        _common = dict(_dtype=_name, _code=_lib.DTYPE_CODE[_name], _non_native=_nn, _itemsize=_isz)
        _make("BinnerScalar_" + _sfx, _BinnerScalar, **_common)
        _make("BinnerOrdinal_" + _sfx, _BinnerOrdinal, **_common)
        if not _nn:
            _make("BinnerHash_" + _sfx, _BinnerHash, **_common)
        for _prefix, _op in _AGG_OPS.items():
            _make(_prefix + "_" + _sfx, Aggregator, _op=_op, **_common)
        _make("AggNUnique_" + _sfx, _AggNUnique, **_common)
        # the reference binds AggList_<dtype>_int64 (src/agg_list.cpp:225-238: the second type is the reserved sort column's)
        _make("AggList_" + _name + "_int64" + ("_non_native" if _nn else ""), _AggList, **_common)
        for _name2 in _DT:
            _make("AggFirst_" + _name + "_" + _name2 + ("_non_native" if _nn else ""), Aggregator, _op=_lib.AGG_FIRST, _dtype2=_name2, **_common)


class AggCount_string(Aggregator):
    """count(string column) = rows whose string is not null, per cell (src/agg_count.cpp:120-160).  The string column is reduced to
    its validity bytes on the host (one byte per row, the arrow bitmap unpacked); the device counts them with the ordinary
    AggCount kernel, the validity doubling as the data mask."""
    _dtype, _code, _non_native, _itemsize, _op = "uint8", _lib.DTYPE_CODE["uint8"], False, 1, _lib.AGG_COUNT

    def set_data(self, thread, ar, index=0):
        from .superutils import string_buffers
        offsets, _, mask = string_buffers(ar)
        n = len(offsets) - 1
        valid = np.ones(n, np.uint8) if mask is None else (1 - mask).astype(np.uint8)
        self._valid = getattr(self, "_valid", {})
        self._valid[int(thread)] = valid
        super().set_data(thread, valid, 0)
        self._string_mask_user = getattr(self, "_string_mask_user", {})
        self._apply_mask(int(thread))

    def _apply_mask(self, thread):
        user = self._string_mask_user.get(thread)
        valid = self._valid.get(thread)
        if valid is None:
            return
        m = valid if user is None else (valid & (np.asarray(user) != 0).astype(np.uint8))
        super().set_data_mask(thread, m)

    def set_data_mask(self, thread, ar):
        self._string_mask_user = getattr(self, "_string_mask_user", {})
        self._string_mask_user[int(thread)] = ar
        self._apply_mask(int(thread))

    def clear_data_mask(self, thread):
        self._string_mask_user = getattr(self, "_string_mask_user", {})
        self._string_mask_user.pop(int(thread), None)
        self._apply_mask(int(thread))


class AggNUnique_string(_AggNUnique):
    """nunique(string column) per cell (src/agg_nunique_string.cpp:10-95: a counter<string> per cell).  Here the strings are first
    encoded by ONE device ordered_set_string (nmaps = 1: a key's ordinal never changes once assigned) and the per-cell distinct
    count runs over the int64 ordinals with the numeric AggNUnique kernel — equal strings have equal ordinals and different
    strings different ones (the string set verifies the bytes behind every hash), so the counts are the reference's."""
    _dtype, _code, _non_native, _itemsize = "int64", _lib.DTYPE_CODE["int64"], False, 8

    def __init__(self, grid, grids, threads, dropmissing=False, dropnan=False):
        super().__init__(grid, grids, threads, dropmissing, dropnan)
        from .superutils import ordered_set_string
        self._strings = ordered_set_string(1)
        self._codes = {}

    def set_data(self, thread, ar, index=0):
        from .superutils import string_buffers
        thread = int(thread)
        _, _, mask = string_buffers(ar)
        self._strings.update(ar)
        codes = self._strings.map_ordinal(ar, slot=thread, device=True)
        self._codes[thread] = codes
        super().set_data(thread, codes, 0)
        n = len(codes)
        self._valid = getattr(self, "_valid", {})
        self._valid[thread] = np.ones(n, np.uint8) if mask is None else (1 - mask).astype(np.uint8)
        self._apply_mask(thread)

    # the task part sets / clears the data mask AFTER set_data (vaex/cpu.py:765-784): the strings' own validity has to survive that
    def _apply_mask(self, thread):
        valid = getattr(self, "_valid", {}).get(thread)
        if valid is None:
            return
        user = getattr(self, "_user_mask", {}).get(thread)
        m = valid if user is None else (valid & (np.asarray(user) != 0).astype(np.uint8))
        super().set_data_mask(thread, m)  # NUNIQUE: mask = 0 marks a null row (include/b200agg.h)

    def set_data_mask(self, thread, ar):
        self._user_mask = getattr(self, "_user_mask", {})
        self._user_mask[int(thread)] = ar
        self._apply_mask(int(thread))

    def clear_data_mask(self, thread):
        getattr(self, "_user_mask", {}).pop(int(thread), None)
        self._apply_mask(int(thread))


class AggList_string_int64(_AggList):
    """``AggList_string_int64(grid, grids, threads, dropnan=False, dropnull=False)`` (src/agg_list.cpp:122-222): per cell the list of the
    rows' strings in arrival order.  A null string stays a null element at its arrival position unless dropnull; dropnan has no
    effect.  REFERENCE QUIRK, kept: the data mask is stored but never read by aggregate() (:183-197), so ``set_data_mask`` — which is
    how a selection reaches an aggregator (vaex/cpu.py:765-784) — filters nothing.  ``get_result()`` returns a pyarrow
    ``large_list<large_string>`` with one list per cell of the full grid (first binner fastest), built from the device's buffers."""
    _op = _lib.AGG_LIST_STRING
    _dtype, _code, _non_native, _itemsize = "uint8", _lib.DTYPE_CODE["uint8"], False, 1

    def set_data(self, thread, strings, index=0):
        """strings: what ``superutils.string_buffers`` takes (pyarrow string / large_string, also sliced or chunked; numpy object
        arrays; lists), or the buffers themselves as ``(int64 offsets[n + 1], uint8 bytes, uint8 null mask or None)``, host (numpy)
        or device (torch CUDA tensors) arrays."""
        from .superutils import string_buffers
        if isinstance(strings, tuple):
            offsets, data, mask = strings
        else:
            offsets, data, mask = string_buffers(strings)
        off = _lib.column(offsets)
        if off.dtype != np.dtype("int64"):
            raise RuntimeError("string offsets must be int64")
        self._data[int(thread)] = (off, _lib.column(data) if len(data) else None, None if mask is None else _lib.mask_column(mask))

    def set_data_mask(self, thread, ar):
        pass  # read by nothing in the reference (src/agg_list.cpp:183-197)

    def clear_data_mask(self, thread):
        pass

    def _fill(self, a, thread):
        buffers = self._data.get(thread)
        if buffers is None:
            raise RuntimeError("string_sequence not set")  # src/agg_list.cpp:185-187
        off, data, mask = buffers
        a.agg = self._h
        a.data = off.ptr
        keep = [off]
        if data is not None:
            a.order = data.ptr
            # the byte buffer is not row-shaped: it joins the memspace decision, not Grid.bin's length check
            keep.append(types.SimpleNamespace(memspace=data.memspace, length=off.length - 1, keep=data))
        if mask is not None:
            a.mask = mask.ptr
            keep.append(mask)
        return keep

    def result_arrays(self):
        """(int64 list offsets[cells + 1], int64 string offsets[n + 1], uint8 bytes, uint8 null flags[n]) of the n elements"""
        nelem, nbytes = C.c_int64(0), C.c_int64(0)
        _lib.check(_lib.lib().b200_agg_list_string_finish(self._h, C.byref(nelem), C.byref(nbytes)))
        list_offsets = np.zeros(len(self.grid) + 1, np.int64)
        str_offsets = np.zeros(nelem.value + 1, np.int64)
        data = np.zeros(max(nbytes.value, 1), np.uint8)
        nulls = np.zeros(max(nelem.value, 1), np.uint8)
        _lib.check(_lib.lib().b200_agg_list_string_read(self._h, list_offsets.ctypes.data, str_offsets.ctypes.data, data.ctypes.data, nulls.ctypes.data))
        return list_offsets, str_offsets, data[:nbytes.value], nulls[:nelem.value]

    def get_result(self):
        import pyarrow as pa
        list_offsets, str_offsets, data, nulls = self.result_arrays()
        n = len(nulls)
        null_count = int(np.count_nonzero(nulls))
        validity = pa.py_buffer(np.packbits(nulls == 0, bitorder="little")) if null_count else None
        values = pa.Array.from_buffers(pa.large_string(), n, [validity, pa.py_buffer(str_offsets), pa.py_buffer(data)], null_count=null_count)
        return pa.LargeListArray.from_arrays(pa.array(list_offsets), values)


# names the B200 path does not provide: list / object aggregators and BinnerCombined's pybind name for unsupported dtypes.
# Accessing them raises instead of silently doing something else.
_UNSUPPORTED_PREFIXES = ("AggCount_object",)


def __getattr__(name):
    if name.startswith(_UNSUPPORTED_PREFIXES):
        raise AttributeError(f"vaex_b200.superagg.{name}: not on the B200 hot path (use the reference CPU implementation)")
    raise AttributeError(name)
