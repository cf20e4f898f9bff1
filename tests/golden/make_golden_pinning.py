"""Generate tests/golden/pinning_golden.npz from the COMPILED, UNMODIFIED reference (oracle/_ref): what the reference returns for
the cases of tests/test_oracle_pinning.py (random binby problems, the first / last mask quirk, the threaded chunk loop, random
minmax columns) and the class names and grid layout its modules expose (tests/test_cpu_abi.py).  The inputs are rebuilt from their
seeds by tests/helpers.py, so only the reference's answers are stored.  Run where the reference sources exist:

    make -C oracle ref && python tests/golden/make_golden_pinning.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref_driver as R  # noqa: E402
import helpers as H  # noqa: E402

RANDOM_SEEDS = 12
MINMAX_SEEDS = 6
MIRRORED_PREFIXES = ("BinnerScalar_", "BinnerOrdinal_", "AggCount_", "AggSum_", "AggSumMoment_", "AggMin_", "AggMax_", "AggFirst_", "AggNUnique_")


def results(out, name, res):
    for k, r in enumerate(res):
        if np.ma.isMaskedArray(r):
            out[f"{name}/a{k}_result"] = np.asarray(r.data)
            out[f"{name}/a{k}_result_mask"] = np.ma.getmaskarray(r)
        else:
            out[f"{name}/a{k}_result"] = np.asarray(r)


def cases():
    out = {}
    for seed in range(RANDOM_SEEDS):
        results(out, f"random_{seed}", R.binby(*H.random_binby_case(seed)))
    results(out, "first_mask_quirk", R.binby(*H.first_mask_quirk_case()))
    b, a, n = H.chunk_loop_case()
    for nthreads in H.CHUNK_LOOP_THREADS:
        results(out, f"chunk_loop_{nthreads}", R.RefBinby(b, a, nthreads).run(n, chunk=H.CHUNK_LOOP_CHUNK))
    for seed in range(MINMAX_SEEDS):
        out[f"minmax_{seed}/raw"] = np.array([R.minmax(col, raw=True) for _, col in H.minmax_random_columns(seed)])
    superagg, superutils = R.modules()
    out["names/superagg"] = np.array(sorted(n for n in dir(superagg) if n.startswith(MIRRORED_PREFIXES) and not n.endswith(("_string", "_object"))))
    out["names/ordered_sets"] = np.array(sorted(n for n in dir(superutils) if n.startswith("ordered_set_") and n not in ("ordered_set_string", "ordered_set_object")))
    rb = H.grid_layout_binners(superagg)
    rg = superagg.Grid(rb)
    out["grid_layout/shapes"] = np.array(list(rg.shapes))
    out["grid_layout/strides"] = np.array(list(rg.strides))
    out["grid_layout/length"] = np.array(len(rg))
    out["grid_layout/binner_lengths"] = np.array([len(b) for b in rb])
    return out


if __name__ == "__main__":
    here = os.path.dirname(os.path.abspath(__file__))
    path = os.path.join(here, "pinning_golden.npz")
    data = cases()
    np.savez_compressed(path, **data)
    print("wrote", len(data), "arrays,", os.path.getsize(path) // 1024, "KiB")
