"""Aggregator descriptors — host-side mirror of ``vaex.agg`` for the binned-statistics path.

Reference: packages/vaex-core/vaex/agg.py:221-335 (AggregatorDescriptorBasic: encode, _prepare_types, _create_operation with the
grid-count heuristic and memory accounting, get_result edge slicing), :386-523 (mean / var / std / skew / kurtosis as
combinations of primitive grids + ``finish``), :525-606 (count, sum, mean, min, max, first, last, std, var, ...).
The primitive aggregations run on the GPU (vaex_b200.superagg); ``finish`` is O(cells) numpy like in the reference.
nunique (vaex/agg.py:338-369, 600-612) and list, on numeric and string columns, run on the device too.  Out of scope here
(SURVEY.md 8f): describe, object columns.
"""
import operator
from functools import reduce

import numpy as np

from . import superagg

_min, _max, _list = min, max, list  # the module defines its own min / max / list, like vaex.agg does


def _upcast(dtype):
    dtype = np.dtype(dtype).newbyteorder("=")
    if dtype.kind == "f":
        return np.dtype("float64")
    if dtype.kind in "ib":
        return np.dtype("int64")
    if dtype.kind == "u":
        return np.dtype("uint64")
    return dtype


def find_type_from_dtype(namespace, prefix, dtype, *others):
    """vaex.utils.find_type_from_dtype (vaex/utils.py:754-791): ``prefix + dtype [+ '_' + dtype2] [+ '_non_native']``."""
    dtype = np.dtype(dtype)
    if dtype.kind in "OU":  # string columns: the reference's classes carry the suffix "string" (+ "_<dtype2>", AggList_string_int64)
        name = prefix + "string"
        for o in others:
            name += "_" + np.dtype(o).newbyteorder("=").name
        if not hasattr(namespace, name):
            raise ValueError(f"Could not find a class ({name}), seems strings are not supported.")
        return getattr(namespace, name)
    if dtype.kind in "mM":
        dtype = np.dtype("int64") if dtype.kind == "m" else np.dtype("uint64")
    name = prefix + dtype.newbyteorder("=").name
    for o in others:
        name += "_" + np.dtype(o).newbyteorder("=").name
    if dtype.byteorder not in ("=", "|") and dtype.byteorder != ("<" if np.little_endian else ">"):
        name += "_non_native"
    if not hasattr(namespace, name):
        raise ValueError(f"Could not find a class ({name}), seems {dtype} is not supported.")
    return getattr(namespace, name)


class AggregatorDescriptor:
    def __repr__(self):
        return "vaex_b200.agg.{}({!r})".format(self.short_name, ", ".join(map(str, self.expressions)))

    def finish(self, value):
        return value


class AggregatorDescriptorBasic(AggregatorDescriptor):
    """One primitive aggregation == one native Agg* object (vaex/agg.py:221-335)."""

    def __init__(self, name, expressions, short_name, agg_args=(), selection=None, edges=False):
        self.name = name
        self.short_name = short_name
        self.agg_args = _list(agg_args)
        self.edges = edges
        self.selection = selection
        self.expressions = [str(k) for k in expressions if k is not None]
        if len(self.expressions) == 1 and self.expressions[0] == "*":
            self.expressions = []

    def encode(self, encoding=None):
        # identical keys to vaex/agg.py:240-252
        spec = {"aggregation": self.short_name}
        if self.expressions:
            spec["expressions"] = _list(self.expressions)
        if self.selection is not None:
            spec["selection"] = self.selection
        if self.edges:
            spec["edges"] = True
        if self.agg_args and self.short_name not in ["first", "last"]:
            spec["parameters"] = self.agg_args
        return spec

    def primitives(self):
        return [self]

    def _prepare_types(self, dtypes):
        """dtypes: mapping expression -> numpy dtype (vaex/agg.py:254-265)."""
        if len(self.expressions) == 0 and self.short_name == "count":
            self.dtypes_in = []
            self.dtype_in = np.dtype("int64")
            self.dtype_out = np.dtype("int64")
        else:
            self.dtypes_in = [np.dtype(dtypes[e]) for e in self.expressions]
            self.dtype_in = self.dtypes_in[0]
            self.dtype_out = self.dtype_in
            if self.short_name == "count":
                self.dtype_out = np.dtype("int64")
            if self.short_name in ["sum", "_sum_moment"]:
                self.dtype_out = _upcast(self.dtype_in)

    def _create_operation(self, grid, nthreads):
        # vaex/agg.py:278-321
        if self.name in ("AggFirst", "AggList"):
            if len(self.dtypes_in) == 1:
                agg_op_type = find_type_from_dtype(superagg, self.name + "_", self.dtypes_in[0], np.dtype("int64"))
            else:
                agg_op_type = find_type_from_dtype(superagg, self.name + "_", self.dtypes_in[0], self.dtypes_in[1])
        else:
            agg_op_type = find_type_from_dtype(superagg, self.name + "_", self.dtype_in)
        ncells = len(grid)
        grids = nthreads
        if ncells >= 1e4:
            grids = _min(32, nthreads)
        if ncells >= 1e5:
            grids = _min(16, nthreads)
        if ncells >= 1e6:
            grids = _min(8, nthreads)
        grids = _max(grids, 1)
        if self.short_name == "list":  # "cannot predict memory usage", grids = 1 (vaex/agg.py:306-309)
            import sys
            agg_op = agg_op_type(grid, 1, nthreads, *self.agg_args)
            self.predicted_memory_usage = sys.getsizeof(agg_op)
            return agg_op
        # memory pre-declaration (vaex/agg.py:309-318): bytes_per_cell * cells * grids is declared before the aggregator exists and
        # must equal what the object then reports
        import sys
        self.predicted_memory_usage = self.dtype_out.itemsize * ncells * grids
        agg_op = agg_op_type(grid, grids, nthreads, *self.agg_args)
        used_memory = agg_op.__sizeof__()
        if used_memory != self.predicted_memory_usage:
            raise RuntimeError(f"Wrong prediction for {agg_op_type}, expected to take {self.predicted_memory_usage} bytes but actually used {used_memory}")
        self.predicted_memory_usage = sys.getsizeof(agg_op)  # what TaskPartAggregation.memory_usage() sums (vaex/cpu.py:649)
        return agg_op

    def get_result(self, agg_operation):
        # vaex/agg.py:323-335: drop the edge cells unless edges=True (scalar [2:-1], ordinal [0:-2])
        grid = agg_operation.get_result()
        if self.short_name == "list":
            return grid  # one list per cell of the FULL grid (edge cells included), flat order, first binner fastest
        if not self.edges:
            def binner2slice(binner):
                name = type(binner).__name__
                if name.startswith("BinnerScalar_"):
                    return slice(2, -1)
                if name.startswith(("BinnerOrdinal_", "BinnerHash_")):
                    return slice(0, -2)
                raise TypeError(f"Binner not supported with edges=False {binner}")
            grid = grid[tuple(binner2slice(b) for b in agg_operation.grid.binners)]
        return grid


class AggregatorDescriptorNUnique(AggregatorDescriptorBasic):
    """vaex/agg.py:338-369: one shared (thread safe) set structure, grids = 1, int64 result."""

    def __init__(self, name, expression, short_name, dropmissing, dropnan, selection=None, edges=False):
        super().__init__(name, expression, short_name, selection=selection, edges=edges)
        self.dropmissing = dropmissing
        self.dropnan = dropnan

    def encode(self, encoding=None):
        spec = super().encode(encoding)
        if self.dropmissing:
            spec["dropmissing"] = self.dropmissing
        if self.dropnan:
            spec["dropnan"] = self.dropnan
        return spec

    def _prepare_types(self, dtypes):
        super()._prepare_types(dtypes)
        self.dtype_out = np.dtype("int64")

    def _create_operation(self, grid, nthreads):
        agg_op_type = find_type_from_dtype(superagg, self.name + "_", self.dtype_in)
        return agg_op_type(grid, 1, nthreads, self.dropmissing, self.dropnan)


class AggregatorDescriptorMulti(AggregatorDescriptor):
    """mean / var / std / skew / kurtosis: several primitive grids + finish() (vaex/agg.py:373-523)."""

    def __init__(self, short_name, expression, selection=None, edges=False, ddof=0):
        self.short_name = short_name
        self.expressions = [str(expression)]
        self.selection = selection
        self.edges = edges
        self.ddof = ddof
        e, kw = self.expressions[0], dict(selection=selection, edges=edges)
        if short_name == "mean":
            self.parts = [sum(e, **kw), count(e, **kw)]
        elif short_name in ("var", "std"):
            self.parts = [_sum_moment(e, 2, **kw), sum(e, **kw), count(e, **kw)]
        elif short_name == "skew":
            self.parts = [_sum_moment(e, 1, **kw), _sum_moment(e, 2, **kw), _sum_moment(e, 3, **kw), count(e, **kw)]
        elif short_name == "kurtosis":
            self.parts = [_sum_moment(e, 1, **kw), _sum_moment(e, 2, **kw), _sum_moment(e, 3, **kw), _sum_moment(e, 4, **kw), count(e, **kw)]
        else:
            raise ValueError(short_name)

    def primitives(self):
        return self.parts

    def combine(self, *grids):
        with np.errstate(divide="ignore", invalid="ignore"):
            if self.short_name == "mean":  # vaex/agg.py:403-418
                s, n = grids
                return np.asarray(s) / n
            if self.short_name in ("var", "std"):  # vaex/agg.py:439-455 — raw moments, NOT Welford (kept for parity)
                m2, s, n = grids
                mean = np.asarray(s) / n
                variance = np.asarray(m2) / n - mean ** 2
                return variance ** 0.5 if self.short_name == "std" else variance
            if self.short_name == "skew":  # vaex/agg.py:474-481
                s1, s2, s3, n = grids
                m1, m2, m3 = s1 / n, s2 / n, s3 / n
                return (m3 - 3 * m1 * m2 + 2 * m1 ** 3) / (m2 - m1 ** 2) ** (3 / 2)
            s1, s2, s3, s4, n = grids  # kurtosis, vaex/agg.py:506-514
            m1, m2, m3, m4 = s1 / n, s2 / n, s3 / n, s4 / n
            return (m4 - 4 * m1 * m3 + 6 * m1 ** 2 * m2 - 3 * m1 ** 4) / (m2 - m1 ** 2) ** 2 - 3.0


def count(expression="*", selection=None, edges=False):
    return AggregatorDescriptorBasic("AggCount", [expression], "count", selection=selection, edges=edges)


def sum(expression, selection=None, edges=False):
    return AggregatorDescriptorBasic("AggSum", [expression], "sum", selection=selection, edges=edges)


def _sum_moment(expression, moment, selection=None, edges=False):
    return AggregatorDescriptorBasic("AggSumMoment", [expression], "_sum_moment", agg_args=[moment], selection=selection, edges=edges)


def min(expression, selection=None, edges=False):
    return AggregatorDescriptorBasic("AggMin", [expression], "min", selection=selection, edges=edges)


def max(expression, selection=None, edges=False):
    return AggregatorDescriptorBasic("AggMax", [expression], "max", selection=selection, edges=edges)


def first(expression, order_expression=None, selection=None, edges=False):
    return AggregatorDescriptorBasic("AggFirst", [expression, order_expression], "first", agg_args=[False], selection=selection, edges=edges)


def last(expression, order_expression=None, selection=None, edges=False):
    return AggregatorDescriptorBasic("AggFirst", [expression, order_expression], "last", agg_args=[True], selection=selection, edges=edges)


def mean(expression, selection=None, edges=False):
    return AggregatorDescriptorMulti("mean", expression, selection=selection, edges=edges)


def var(expression, ddof=0, selection=None, edges=False):
    return AggregatorDescriptorMulti("var", expression, selection=selection, edges=edges, ddof=ddof)


def std(expression, ddof=0, selection=None, edges=False):
    return AggregatorDescriptorMulti("std", expression, selection=selection, edges=edges, ddof=ddof)


def skew(expression, selection=None, edges=False):
    return AggregatorDescriptorMulti("skew", expression, selection=selection, edges=edges)


def kurtosis(expression, selection=None, edges=False):
    return AggregatorDescriptorMulti("kurtosis", expression, selection=selection, edges=edges)


def from_spec(spec):
    """Decode vaex's aggregation spec dict (vaex/agg.py:240-252 encode) back into a descriptor."""
    name = spec["aggregation"]
    exprs = spec.get("expressions", ["*"])
    kw = dict(selection=spec.get("selection"), edges=spec.get("edges", False))
    if name == "count":
        return count(exprs[0] if exprs else "*", **kw)
    if name == "sum":
        return sum(exprs[0], **kw)
    if name == "_sum_moment":
        return _sum_moment(exprs[0], spec["parameters"][0], **kw)
    if name == "min":
        return min(exprs[0], **kw)
    if name == "max":
        return max(exprs[0], **kw)
    if name in ("first", "last"):
        f = first if name == "first" else last
        return f(exprs[0], exprs[1] if len(exprs) > 1 else None, **kw)
    if name == "nunique":
        return nunique(exprs[0], dropnan=spec.get("dropnan", False), dropmissing=spec.get("dropmissing", False), **kw)
    if name == "list":
        params = spec.get("parameters", [False, False])
        return list(exprs[0], dropnan=params[0], dropmissing=params[1], **kw)
    raise ValueError(f"aggregation {name!r} is not on the B200 hot path")


def list(expression, selection=None, dropna=False, dropnan=False, dropmissing=False, edges=False):
    """Aggregator that returns the list of values per bin (vaex/agg.py:654-674 -> AggList_<dtype>_int64, src/agg_list.cpp)."""
    if dropna:
        dropnan = dropmissing = True
    return AggregatorDescriptorBasic("AggList", [expression], "list", agg_args=[dropnan, dropmissing], selection=selection, edges=edges)


def nunique(expression, dropna=False, dropnan=False, dropmissing=False, selection=None, edges=False):
    """Number of unique items per bin (vaex/agg.py:600-612)."""
    if dropna:
        dropnan = True
        dropmissing = True
    return AggregatorDescriptorNUnique("AggNUnique", [expression], "nunique", dropmissing, dropnan, selection=selection, edges=edges)


aggregates = {f.__name__: f for f in (count, sum, min, max, first, last, mean, var, std, skew, kurtosis, nunique, list)}
