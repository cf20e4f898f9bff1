"""Generate tests/golden/agglist_string_golden.npz from the COMPILED, UNMODIFIED reference (oracle/_ref/superagg*.so):
AggList_string_int64 (src/agg_list.cpp:122-222), driven through the StringList64 glue of oracle/ref_strlist_shim.cpp.  Run where
/root/reference exists:

    make -C oracle -f strlist.mk ref && python tests/golden/make_golden_agglist_string.py

Two binner setups, each fed in several bin() calls: an ordinal binner over -1..ncat+1 (both edge cells) in four calls (one of 0 rows,
one of nulls only, two longer than 1024 rows) and a scalar float64 binner with NaN and out-of-range values in two calls.  Each is run
for dropnull x dropnan x (no data mask, an all-zero data mask).  Strings are 0 to ~3000 bytes, empty ones and non-ASCII UTF-8
included, about 15 % null.  get_result() of the reference hands (offsets, StringList64) to vaex.arrow.convert.list_from_arrays; vaex
cannot be imported here, so a stub module with that one function (returning the buffers) stands in for it.  The archive is written
with fixed member timestamps, so a rerun reproduces it byte for byte."""
import importlib
import io
import os
import sys
import types
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_driver as R  # noqa: E402

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "agglist_string_golden.npz")
ALPHABET = ["a", "b", "z", "Q", " ", "0", "é", "ß", "日本", "€", "😀"]


def make_strings(rng, n, null_rate=0.15):
    """n strings: mostly 1-40 characters, 1 % long (~600-3000 bytes), 5 % empty; -> (offsets, bytes, null mask)"""
    out = []
    for _ in range(n):
        r = rng.random()
        k = 0 if r < 0.05 else int(rng.integers(300, 1400)) if r < 0.06 else int(rng.integers(1, 40))
        out.append("".join(rng.choice(ALPHABET, k)) if k else "")
    enc = [s.encode("utf8") for s in out]
    offsets = np.zeros(n + 1, np.int64)
    offsets[1:] = np.cumsum([len(e) for e in enc])
    nulls = (rng.random(n) < null_rate).astype(np.uint8)
    return offsets, np.frombuffer(b"".join(enc), np.uint8).copy(), nulls


def cases(rng):
    """-> [(name, binner factory, key column, calls, (offsets, bytes, nulls))]"""
    n1, ncat = 3000, 5
    x1 = rng.integers(-1, ncat + 2, n1).astype("i8")
    s1 = make_strings(rng, n1)
    calls1 = [(0, 1100), (1100, 1100), (1100, 1300), (1300, n1)]
    s1[2][1100:1300] = 1  # a call of nulls only
    n2 = 2100
    x2 = rng.uniform(-1.5, 11.5, n2)
    x2[rng.random(n2) < 0.05] = np.nan
    s2 = make_strings(rng, n2)
    return [("ordinal", lambda sa: sa.BinnerOrdinal_int64(1, "x", ncat, 0, False, False), x1, calls1, s1),
            ("scalar", lambda sa: sa.BinnerScalar_float64(1, "x", 0.0, 10.0, 7), x2, [(0, 1030), (1030, n2)], s2)]


def save(path, arrays):
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_DEFLATED) as z:
        for name in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asarray(arrays[name]), allow_pickle=False)
            z.writestr(zipfile.ZipInfo(name + ".npy", date_time=(1980, 1, 1, 0, 0, 0)), buf.getvalue(), compress_type=zipfile.ZIP_DEFLATED)


def main():
    sa, _ = R.modules()
    sys.path.insert(0, R._REF)
    try:
        shim = importlib.import_module("strlist_shim")
    finally:
        sys.path.remove(R._REF)
    vaex, arrow, convert = types.ModuleType("vaex"), types.ModuleType("vaex.arrow"), types.ModuleType("vaex.arrow.convert")
    convert.list_from_arrays = lambda offsets, sl: (np.array(offsets, np.int64),) + tuple(shim.to_numpy(sl))
    vaex.arrow, arrow.convert = arrow, convert
    sys.modules.update({"vaex": vaex, "vaex.arrow": arrow, "vaex.arrow.convert": convert})
    rng = np.random.default_rng(2024)
    out = {}
    for name, make_binner, x, calls, (offsets, data, nulls) in cases(rng):
        out[f"{name}/x"], out[f"{name}/calls"] = x, np.array(calls, np.int64)
        out[f"{name}/offsets"], out[f"{name}/bytes"], out[f"{name}/nulls"] = offsets, data, nulls
        for masked in (False, True):
            for dropnan in (False, True):
                for dropnull in (False, True):
                    b = make_binner(sa)
                    g = sa.Grid([b])
                    a = sa.AggList_string_int64(g, 1, 1, dropnan, dropnull)
                    keep = []
                    for i1, i2 in calls:
                        xs = np.ascontiguousarray(x[i1:i2])
                        sl = shim.string_list(offsets[i1:i2 + 1], data, nulls[i1:i2].copy())
                        keep += [xs, sl]
                        b.set_data(0, xs)
                        a.set_data(0, sl, 0)
                        if masked:  # the data mask a selection arrives as (vaex/cpu.py:765-784): all zero, and read by nothing
                            m = np.zeros(i2 - i1, np.uint8)
                            keep.append(m)
                            a.set_data_mask(0, m)
                        g.bin(0, [a], i2 - i1)
                    res = a.get_result()
                    case = f"{name}/{'masked' if masked else 'plain'}_dropnan{int(dropnan)}_dropnull{int(dropnull)}"
                    for field, arr in zip(("list_offsets", "str_offsets", "out_bytes", "out_nulls"), res):
                        out[f"{case}/{field}"] = np.asarray(arr)
    save(PATH, out)
    print(f"wrote {PATH}: {len(out)} arrays")


if __name__ == "__main__":
    main()
