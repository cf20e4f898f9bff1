"""AggList_string_int64 on the device (csrc/list.cu): time the append (b200_bin) and the finish (sort / offsets + byte gather) of
agg.list on a string column, device-resident, and check a sample against the compiled reference.

    python tools/bench_list_string.py [--rows 100000000] [--groups 1000,1000000] [--repeats 3]

Inputs are seeded and generated on the device: an int64 group code per row (ordinal binner) and strings of 0-24 random letters
(12 B on average), 5 % null.  Times are CUDA events on the slot streams the work runs on, after one untimed warm-up of the same
shape (the aggregator is reset between passes, so the timed passes reuse its buffers).  The finish is timed twice: the first
call sorts the records and builds the result, the second one (nothing new appended) only builds it — the sort is the difference.
Bytes per row are what the algorithm has to move (see `algorithmic_bytes`), against the HBM peak bench.py quotes.  The parity check
runs the first --parity-rows rows through the compiled, unmodified reference (oracle/_ref, built by `make -C oracle -f strlist.mk
ref`) and compares the four result buffers; the reference's own time on that sample gives its rows/s on one host thread (its list
aggregator keeps one shared grid).  One JSON line is printed."""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def algorithmic_bytes(rows, nelem, nbytes, passes):
    """bytes the append and the finish have to move (records are {u64 key, u64 payload} + one u64 pool position per row)"""
    append = rows * (8 + 8 + 1 + 8 + 8 + 8) + 2 * nbytes  # code, offset, null flag, record key/payload/position; bytes in + out of the pool
    sort = passes * rows * (8 + 32)  # per pass: the histogram reads the keys, the scatter reads and writes key + payload
    build = rows * 8 + nelem * (2 * (8 + 16) + 8 + 1) + nelem * (8 + 16 + 8) + 2 * nbytes  # counts; 2 length passes + offsets + flags; gather
    return append, sort, build


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


def make_inputs(rows, groups, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    codes = torch.randint(0, groups, (rows,), device="cuda", generator=g, dtype=torch.int64)
    lengths = torch.randint(0, 25, (rows,), device="cuda", generator=g, dtype=torch.int64)
    offsets = torch.zeros(rows + 1, device="cuda", dtype=torch.int64)
    torch.cumsum(lengths, 0, out=offsets[1:])
    nbytes = int(offsets[-1])
    data = torch.randint(97, 123, (max(nbytes, 1),), device="cuda", generator=g, dtype=torch.uint8)
    nulls = (torch.rand(rows, device="cuda", generator=g) < 0.05).to(torch.uint8)
    return codes, offsets, data, nulls


def run_device(codes, offsets, data, nulls, groups, repeats):
    import torch
    from vaex_b200 import _lib, superagg
    rows = codes.numel()
    b = superagg.BinnerOrdinal_int64(1, "code", groups, 0, False, False)
    grid = superagg.Grid([b])
    a = superagg.AggList_string_int64(grid, 1, 1)
    b.set_data(0, codes)
    a.set_data(0, (offsets, data, nulls))
    stream = torch.cuda.ExternalStream(a._ctx.stream(0))
    nelem, nbytes = C.c_int64(0), C.c_int64(0)

    def finish():
        _lib.check(_lib.lib().b200_agg_list_string_finish(a._h, C.byref(nelem), C.byref(nbytes)))

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)

    out = {"append_ms": [], "finish_ms": [], "rebuild_ms": []}
    for rep in range(repeats + 1):  # pass 0 warms up
        a.reset()
        torch.cuda.synchronize()
        t_append = timed(lambda: grid.bin(0, [a], rows))
        t_finish = timed(finish)
        t_rebuild = timed(finish)
        if rep:
            out["append_ms"].append(t_append)
            out["finish_ms"].append(t_finish)
            out["rebuild_ms"].append(t_rebuild)
    med = {k: float(np.median(v)) for k, v in out.items()}
    return med, nelem.value, nbytes.value, a


def reference_parity(codes, offsets, data, nulls, groups, sample, device_agg_factory):
    """the first `sample` rows through the compiled reference and through the device; -> (equal, reference rows/s)"""
    from oracle import ref_driver as R
    if not R.available():
        return None, None, "compiled reference missing (make -C oracle -f strlist.mk ref)"
    sa, _ = R.modules()
    sys.path.insert(0, R._REF)
    try:
        shim = importlib.import_module("strlist_shim")
    except ImportError:
        return None, None, "oracle/_ref/strlist_shim missing (make -C oracle -f strlist.mk ref)"
    finally:
        sys.path.remove(R._REF)
    vaex, arrow, convert = types.ModuleType("vaex"), types.ModuleType("vaex.arrow"), types.ModuleType("vaex.arrow.convert")
    convert.list_from_arrays = lambda o, sl: (np.array(o, np.int64),) + tuple(shim.to_numpy(sl))
    vaex.arrow, arrow.convert = arrow, convert
    sys.modules.update({"vaex": vaex, "vaex.arrow": arrow, "vaex.arrow.convert": convert})
    x = codes[:sample].cpu().numpy()
    off = offsets[:sample + 1].cpu().numpy()
    by = data[:int(off[-1])].cpu().numpy()
    nu = nulls[:sample].cpu().numpy()
    b = sa.BinnerOrdinal_int64(1, "code", groups, 0, False, False)
    g = sa.Grid([b])
    a = sa.AggList_string_int64(g, 1, 1, False, False)
    sl = shim.string_list(off, by, nu)
    b.set_data(0, x)
    a.set_data(0, sl, 0)
    t0 = time.perf_counter()
    g.bin(0, [a], sample)
    want = a.get_result()
    dt = time.perf_counter() - t0
    got = device_agg_factory(x, off, by, nu)
    equal = all(w.dtype == h.dtype and np.array_equal(w, h) for w, h in zip(want, got))
    return equal, sample / dt, "compiled reference, 1 host thread, bin() + get_result()"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=float, default=1e8)
    ap.add_argument("--groups", default="1000,1000000")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--parity-rows", type=float, default=1e6)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_list_string.py needs a CUDA device")
    import bench
    from vaex_b200 import superagg
    rows, sample = int(args.rows), int(args.parity_rows)
    peak, peak_src = bench.measured_peak()
    name, power = gpu_info()
    result = {"bench": "agg_list_string", "gpu": name, "power_limit": power, "rows": rows, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "configs": []}
    parity_all = True
    for groups in [int(g) for g in args.groups.split(",")]:
        codes, offsets, data, nulls = make_inputs(rows, groups, seed=groups)
        med, nelem, nbytes, _ = run_device(codes, offsets, data, nulls, groups, args.repeats)
        cells = groups + 2
        passes = (int(cells).bit_length() + 7) // 8
        append_b, sort_b, build_b = algorithmic_bytes(rows, nelem, nbytes, passes)
        sort_ms = med["finish_ms"] - med["rebuild_ms"]

        def device_sample(x, off, by, nu):
            b = superagg.BinnerOrdinal_int64(1, "code", groups, 0, False, False)
            g = superagg.Grid([b])
            a = superagg.AggList_string_int64(g, 1, 1)
            b.set_data(0, x)
            a.set_data(0, (off, by, nu))
            g.bin(0, [a], len(x))
            return a.result_arrays()
        equal, ref_rps, ref_note = reference_parity(codes, offsets, data, nulls, groups, sample, device_sample)
        parity_all = parity_all and bool(equal)
        total_ms = med["append_ms"] + med["finish_ms"]
        gbs = lambda b, ms: b / (ms * 1e-3) / 1e9 if ms > 0 else None
        result["configs"].append({
            "groups": groups, "elements": nelem, "bytes": nbytes, "radix_passes": passes,
            "append_ms": round(med["append_ms"], 3), "finish_ms": round(med["finish_ms"], 3),
            "finish_sort_ms": round(sort_ms, 3), "finish_offsets_gather_ms": round(med["rebuild_ms"], 3),
            "rows_per_s": rows / (total_ms * 1e-3),
            "algorithmic_bytes_per_row": {"append": append_b / rows, "sort": sort_b / rows, "offsets_gather": build_b / rows},
            "append_hbm_fraction": gbs(append_b, med["append_ms"]) / peak, "sort_hbm_fraction": gbs(sort_b, sort_ms) / peak if sort_ms > 0 else None,
            "offsets_gather_hbm_fraction": gbs(build_b, med["rebuild_ms"]) / peak,
            "end_to_end_hbm_fraction": gbs(append_b + sort_b + build_b, total_ms) / peak,
            "parity_rows": sample, "parity": equal, "reference_rows_per_s": ref_rps, "reference": ref_note,
        })
        del codes, offsets, data, nulls
        torch.cuda.empty_cache()
    result["parity"] = parity_all
    print(json.dumps(result))


if __name__ == "__main__":
    main()
