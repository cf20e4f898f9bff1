"""Shared helpers: run the same spec dicts (oracle.scalar/ordinal/agg) through the product (vaex_b200.superagg)."""
import numpy as np


def _suffix(ar):
    ar = np.asarray(ar) if not hasattr(ar, "__cuda_array_interface__") or isinstance(ar, np.ndarray) else ar
    dt = np.dtype(ar.dtype) if isinstance(ar, np.ndarray) else np.dtype(str(ar.dtype).replace("torch.", ""))
    name = dt.newbyteorder("=").name
    swapped = dt.byteorder not in ("=", "|") and dt.byteorder != ("<" if np.little_endian else ">")
    return name + ("_non_native" if swapped else "")


def to_device(ar):
    """numpy -> torch CUDA tensor (byte-swapped arrays are shipped as their raw native-typed bytes)."""
    import torch
    if ar is None:
        return None
    ar = np.ascontiguousarray(ar)
    if ar.dtype == np.bool_:
        return torch.from_numpy(ar).cuda()
    if ar.dtype.kind == "u" and ar.dtype.itemsize > 1:
        # torch has limited unsigned support: move the bytes as the signed type of equal width
        return torch.from_numpy(ar.view(ar.dtype.newbyteorder("=").str.replace("u", "i"))).cuda()
    return torch.from_numpy(ar.view(ar.dtype.newbyteorder("="))).cuda()


class B200Binby:
    """The product-side twin of oracle.ref_driver.RefBinby: same class names, same call protocol."""

    def __init__(self, binners, aggs, nthreads=1):
        from vaex_b200 import superagg
        self.binner_specs, self.agg_specs, self.nthreads = binners, aggs, nthreads
        self.binners = []
        for b in binners:
            sfx = _suffix(b["data"])
            if b["kind"] == "scalar":
                self.binners.append(getattr(superagg, "BinnerScalar_" + sfx)(nthreads, "x", b["vmin"], b["vmax"], b["bins"]))
            elif b["kind"] == "ordinal":
                self.binners.append(getattr(superagg, "BinnerOrdinal_" + sfx)(nthreads, "x", b["count"], b["min_value"], b["allow_other"], b["invert"]))
            else:
                self.binners.append(getattr(superagg, "BinnerHash_" + sfx)(nthreads, "x", b["set"], b.get("allow_other", False), b.get("invert", False)))
        self.grid = superagg.Grid(self.binners)
        self.aggs = []
        for a in aggs:
            op, data = a["op"], a["data"]
            sfx = "int64" if data is None else _suffix(data)
            if op == "count":
                agg = getattr(superagg, "AggCount_" + sfx)(self.grid, 1, nthreads)
            elif op == "sum":
                agg = getattr(superagg, "AggSum_" + sfx)(self.grid, 1, nthreads)
            elif op == "sum_moment":
                agg = getattr(superagg, "AggSumMoment_" + sfx)(self.grid, 1, nthreads, a["moment"])
            elif op == "min":
                agg = getattr(superagg, "AggMin_" + sfx)(self.grid, 1, nthreads)
            elif op == "max":
                agg = getattr(superagg, "AggMax_" + sfx)(self.grid, 1, nthreads)
            elif op in ("first", "last"):
                order = a.get("order")
                sfx2 = "int64" if order is None else np.asarray(order).dtype.newbyteorder("=").name
                name = "AggFirst_" + np.asarray(data).dtype.newbyteorder("=").name + "_" + sfx2 + ("_non_native" if sfx.endswith("_non_native") else "")
                agg = getattr(superagg, name)(self.grid, 1, nthreads, op == "last")
            elif op == "nunique":
                agg = getattr(superagg, "AggNUnique_" + sfx)(self.grid, 1, nthreads, a.get("dropmissing", False), a.get("dropnan", False))
            else:
                raise ValueError(op)
            self.aggs.append(agg)

    def process(self, thread, i1, i2, device=False):
        conv = to_device if device else (lambda x: x)
        sl = slice(i1, i2)
        for binner, spec in zip(self.binners, self.binner_specs):
            binner.set_data(thread, conv(np.asarray(spec["data"])[sl]))
            if spec.get("mask") is not None:
                binner.set_data_mask(thread, conv(np.asarray(spec["mask"])[sl]))
            else:
                binner.clear_data_mask(thread)
        for agg, spec in zip(self.aggs, self.agg_specs):
            if spec["data"] is not None:
                agg.set_data(thread, conv(np.asarray(spec["data"])[sl]), 0)
            if spec.get("order") is not None:
                agg.set_data(thread, conv(np.asarray(spec["order"])[sl]), 1)
            if spec["mask"] is not None:
                agg.set_data_mask(thread, conv(np.asarray(spec["mask"])[sl]))
            else:
                agg.clear_data_mask(thread)
            if spec["op"] == "nunique":
                if spec.get("selection") is not None:
                    agg.set_selection_mask(thread, conv(np.asarray(spec["selection"])[sl]))
                else:
                    agg.clear_selection_mask(thread)
        self.grid.bin(thread, self.aggs, i2 - i1, row_offset=i1)

    def run(self, length, chunk=None, device=False):
        chunk = chunk or max(length, 1)
        t = 0
        for i1 in range(0, length, chunk):
            self.process(t % self.nthreads, i1, min(i1 + chunk, length), device)
            t += 1
        return [a.get_result() for a in self.aggs]


def b200_binby(binners, aggs, length=None, chunk=None, device=False, nthreads=1):
    if length is None:
        length = len(binners[0]["data"])
    return B200Binby(binners, aggs, nthreads).run(length, chunk, device)


def same(a, b, rtol=0.0):
    """bit-exact for integers / min / max / counts; rtol for floating sums."""
    if np.ma.isMaskedArray(a) or np.ma.isMaskedArray(b):
        ma, mb = np.ma.getmaskarray(a), np.ma.getmaskarray(b)
        return np.array_equal(ma, mb) and same(np.asarray(a.data)[~ma], np.asarray(b.data)[~mb], rtol)
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if rtol and a.dtype.kind == "f":
        return np.allclose(a, b, rtol=rtol, atol=0, equal_nan=True)
    return np.array_equal(a, b, equal_nan=a.dtype.kind == "f")


def random_case(rng, n, allow_first=True, float_sum_ok=True):
    """One random (binners, aggs) problem covering every dtype, masks, NaNs, byte order, all aggregators."""
    from oracle import oracle as O
    nd = int(rng.integers(1, 4))
    binners = []
    for d in range(nd):
        if rng.random() < 0.6:
            dt = rng.choice(["f8", "f4", "i8", "i4", "i2", "i1", "u8", "u4", "u2", "u1", "?", ">f8", ">f4", ">i4", ">u2"])
            if np.dtype(dt).kind == "f":
                data = rng.normal(0, 1, n).astype(dt)
                data[rng.random(n) < 0.01] = np.nan
            elif dt == "?":
                data = rng.integers(0, 2, n).astype(dt)
            else:
                data = rng.integers(-5 if np.dtype(dt).kind == "i" else 0, 20, n).astype(dt)
            mask = (rng.random(n) < 0.1) if rng.random() < 0.5 else None
            binners.append(O.scalar(data, -2.5, 3.1, int(rng.integers(1, 12)), mask=mask))
        else:
            dt = rng.choice(["i8", "i4", "i2", "i1", "u8", "u4", "u2", "u1", "?", "f8", "f4", ">i4", ">i8"])
            if np.dtype(dt).kind == "f":
                data = rng.integers(-3, 12, n).astype(dt)
                data[rng.random(n) < 0.02] = np.nan
            elif dt == "?":
                data = rng.integers(0, 2, n).astype(dt)
            else:
                data = rng.integers(-3 if np.dtype(dt).kind == "i" else 0, 12, n).astype(dt)
            mask = (rng.random(n) < 0.1) if rng.random() < 0.5 else None
            binners.append(O.ordinal(data, int(rng.integers(1, 9)), int(rng.integers(-2, 3)), bool(rng.integers(0, 2)), bool(rng.integers(0, 2)), mask=mask))
    aggs = []
    ops = ["count", "count*", "sum", "sum_moment", "min", "max"] + (["first", "last"] if allow_first else [])
    for k in range(int(rng.integers(1, 5))):
        op = rng.choice(ops)
        dt = rng.choice(["f8", "f4", "i8", "i4", "i2", "i1", "u8", "u4", "u2", "u1", "?", ">f8", ">i4"])
        if np.dtype(dt).kind == "f":
            data = rng.normal(0, 10, n).astype(dt)
            data[rng.random(n) < 0.02] = np.nan
        elif dt == "?":
            data = rng.integers(0, 2, n).astype(dt)
        else:
            data = rng.integers(-50 if np.dtype(dt).kind == "i" else 0, 100, n).astype(dt)
        mask = (rng.random(n) < 0.8).astype("u1") if rng.random() < 0.5 else None
        if op == "count*":
            aggs.append(O.agg("count", None, mask))
        elif op == "sum_moment":
            aggs.append(O.agg(op, data, mask, moment=int(rng.integers(0, 5))))
        elif op in ("first", "last"):
            order = None
            if rng.random() < 0.7:
                odt = rng.choice(["f8", "i8", "i4", "u2", "f4"])
                order = rng.normal(0, 100, n).astype(odt) if np.dtype(odt).kind == "f" else rng.integers(0, 1000, n).astype(odt)
            aggs.append(O.agg(op, data, mask, order=order))
        else:
            aggs.append(O.agg(op, data, mask))
    return binners, aggs


# ---- cases pinned to the compiled reference in tests/golden/pinning_golden.npz (tests/golden/make_golden_pinning.py) -----------
def random_binby_case(seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(1, 5000))
    binners, aggs = random_case(rng, n)
    return binners, aggs, n


def first_mask_quirk_case():
    """first / last past 1024 rows with a data mask: AggFirst indexes its mask inside the 1024-row block without the block offset
    (src/agg_first.cpp:131)"""
    from oracle import oracle as O
    rng = np.random.default_rng(77)
    n = 3000
    x = rng.uniform(0, 4, n)
    v = rng.normal(0, 1, n)
    o = rng.integers(0, 100, n).astype("i8")
    m = (rng.random(n) < 0.6).astype("u1")
    return [O.scalar(x, 0, 4, 4)], [O.agg("first", v, m, order=o), O.agg("last", v, m, order=o)], n


CHUNK_LOOP_THREADS = (1, 4)
CHUNK_LOOP_CHUNK = 50_000


def chunk_loop_case():
    from oracle import oracle as O
    rng = np.random.default_rng(5)
    n = 300_000
    x = rng.normal(0, 1, n).astype("f4")
    y = rng.normal(0, 1, n).astype("f4")
    return [O.scalar(x, -3, 3, 64), O.scalar(y, -3, 3, 64)], [O.agg("count")], n


MINMAX_RANDOM_DTYPES = ("f8", "f4", "i8", "i4", "i2", "i1", "u8", "u4", "u2", "u1", "?", ">f8", ">i4", ">u2")


def minmax_random_columns(seed):
    """(dtype, column) pairs for df.minmax: every dtype of MINMAX_RANDOM_DTYPES plain, then half masked"""
    rng = np.random.default_rng(4000 + seed)
    n = int(rng.integers(1, 20000))
    out = []
    for dt in MINMAX_RANDOM_DTYPES:
        d = np.dtype(dt)
        if d.kind == "f":
            v = (rng.standard_normal(n) * 10.0 ** int(rng.integers(-3, 6))).astype(d)
            v[rng.random(n) < 0.2] = np.nan
        elif d.kind == "b":
            v = rng.integers(0, 2, n).astype(d)
        else:
            info = np.iinfo(d)
            v = rng.integers(info.min, info.max, n, dtype=np.int64 if d.kind == "i" else np.uint64, endpoint=True).astype(d)
        out += [(dt, v), (dt, np.ma.array(v, mask=rng.random(n) < 0.5))]
    return out


def grid_layout_binners(superagg):
    """a scalar, an ordinal and an ordinal-with-other binner of `superagg` (the reference's module or the mirror)"""
    return [superagg.BinnerScalar_float64(1, "x", 0, 1, 5), superagg.BinnerOrdinal_int32(1, "y", 4, 0, False, False),
            superagg.BinnerOrdinal_int8(1, "z", 3, 0, True, False)]
