"""tests/golden/agglist_string_golden.npz (tests/golden/make_golden_agglist_string.py) and the two binner setups it was made with."""
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "agglist_string_golden.npz")
FIELDS = ("list_offsets", "str_offsets", "out_bytes", "out_nulls")


def load():
    """setup name -> dict(x, calls, offsets, bytes, nulls, cases={case: dict(masked, dropnan, dropnull, expected=4 arrays)})"""
    z = np.load(PATH, allow_pickle=False)
    out = {}
    for name in ("ordinal", "scalar"):
        s = dict(x=z[f"{name}/x"], calls=[tuple(c) for c in z[f"{name}/calls"].tolist()], offsets=z[f"{name}/offsets"], bytes=z[f"{name}/bytes"],
                 nulls=z[f"{name}/nulls"], cases={})
        for key in z.files:
            if key.startswith(name + "/") and key.endswith("/list_offsets"):
                case = key.split("/")[1]
                s["cases"][case] = dict(masked=case.startswith("masked"), dropnan="dropnan1" in case, dropnull="dropnull1" in case,
                                        expected=tuple(z[f"{name}/{case}/{f}"] for f in FIELDS))
        out[name] = s
    return out


def oracle_binner(name, x):
    from oracle import oracle as O
    return O.ordinal(x, 5, 0) if name == "ordinal" else O.scalar(x, 0.0, 10.0, 7)


def device_binner(name):
    from vaex_b200 import superagg
    return superagg.BinnerOrdinal_int64(1, "x", 5, 0, False, False) if name == "ordinal" else superagg.BinnerScalar_float64(1, "x", 0.0, 10.0, 7)
