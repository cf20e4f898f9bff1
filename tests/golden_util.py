"""Load tests/golden/binstats_golden.npz (generated from the compiled reference by tests/golden/make_golden.py)."""
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "binstats_golden.npz")


def load():
    z = np.load(PATH, allow_pickle=False)
    cases = {}
    for key in z.files:
        name, field = key.split("/", 1)
        cases.setdefault(name, {})[field] = z[key]
    return cases


def binby_case(c):
    """-> (binners, aggs, n, expected) in the oracle's spec-dict form."""
    from oracle import oracle as O
    n = int(c["n"])
    binners, aggs, expected = [], [], []
    for i in range(int(c["nb"])):
        data = c[f"b{i}_data"].view(np.dtype(str(c[f"b{i}_dtype"])))  # restore byte order
        mask = c.get(f"b{i}_mask")
        if str(c[f"b{i}_kind"]) == "scalar":
            binners.append(O.scalar(data, float(c[f"b{i}_vmin"]), float(c[f"b{i}_vmax"]), int(c[f"b{i}_bins"]), mask=mask))
        else:
            binners.append(O.ordinal(data, int(c[f"b{i}_count"]), int(c[f"b{i}_min_value"]), bool(c[f"b{i}_allow_other"]), bool(c[f"b{i}_invert"]), mask=mask))
    for k in range(int(c["na"])):
        data = c.get(f"a{k}_data")
        if data is not None:
            data = data.view(np.dtype(str(c[f"a{k}_dtype"])))
        moment = int(c[f"a{k}_moment"]) if f"a{k}_moment" in c else None
        drop = c.get(f"a{k}_drop", [False, False])
        aggs.append(O.agg(str(c[f"a{k}_op"]), data, c.get(f"a{k}_mask"), moment=moment, order=c.get(f"a{k}_order"), selection=c.get(f"a{k}_selection"),
                          dropmissing=bool(drop[0]), dropnan=bool(drop[1])))
        r = c[f"a{k}_result"]
        if f"a{k}_result_mask" in c:
            r = np.ma.array(r, mask=c[f"a{k}_result_mask"])
        expected.append(r)
    return binners, aggs, n, expected


MINMAX_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "minmax_golden.npz")


def load_minmax():
    """tests/golden/minmax_golden.npz (tests/golden/make_golden_minmax.py): name -> (column incl. byte order / mask, raw (min, max)
    doubles of the compiled reference's statistic grid, the pair cast back to the column dtype)."""
    z = np.load(MINMAX_PATH, allow_pickle=False)
    out = {}
    for name in sorted({k.split("/")[0] for k in z.files}):
        dt = np.dtype(str(z[name + "/dtype"]))
        data = z[name + "/data"].view(dt) if dt.itemsize > 1 else z[name + "/data"]
        if name + "/mask" in z.files:
            data = np.ma.array(data, mask=z[name + "/mask"])
        out[name] = (data, z[name + "/raw"], z[name + "/result"])
    return out


STRINGS_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "strings_golden.npz")


def unpack_strings(offsets, data, nulls=None):
    return [None if (nulls is not None and len(nulls) and nulls[i]) else bytes(data[offsets[i]:offsets[i + 1]]).decode("utf8") for i in range(len(offsets) - 1)]


def load_strings():
    """tests/golden/strings_golden.npz (tests/golden/make_golden_strings.py): name -> dict of arrays"""
    z = np.load(STRINGS_PATH, allow_pickle=False)
    cases = {}
    for key in z.files:
        name, field = key.split("/", 1)
        cases.setdefault(name, {})[field] = z[key]
    return cases


PINNING_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pinning_golden.npz")


def load_pinning():
    """tests/golden/pinning_golden.npz (tests/golden/make_golden_pinning.py): name -> dict of arrays"""
    z = np.load(PINNING_PATH, allow_pickle=False)
    cases = {}
    for key in z.files:
        name, field = key.split("/", 1)
        cases.setdefault(name, {})[field] = z[key]
    return cases


def pinned_results(c):
    """the a<k>_result (+ a<k>_result_mask) arrays of a pinning case -> the reference's result list (numpy.ma where masked)"""
    out = []
    while f"a{len(out)}_result" in c:
        k = len(out)
        r = c[f"a{k}_result"]
        out.append(np.ma.array(r, mask=c[f"a{k}_result_mask"]) if f"a{k}_result_mask" in c else r)
    return out


AGGLIST_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "agglist_golden.npz")


def load_agglist():
    """tests/golden/agglist_golden.npz (tests/golden/make_golden_agglist.py): the shared key column `x` (ordinal binner, `ncat`
    categories), the row where the second bin() call starts (`cut`), per dtype the value column and the data mask, and per case
    ('<dtype>/<plain|masked>_dropnan<0|1>_dropnull<0|1>') the (offsets, values) the compiled reference's AggList returned."""
    z = np.load(AGGLIST_PATH, allow_pickle=False)
    cases = {}
    for key in z.files:
        if key.endswith("/offsets"):
            dt, case, _ = key.split("/")
            cases[f"{dt}/{case}"] = dict(dtype=dt, masked=case.startswith("masked"), dropnan="dropnan1" in case, dropnull="dropnull1" in case,
                                         offsets=z[key], values=z[f"{dt}/{case}/values"], v=z[f"{dt}/v"], valid=z[f"{dt}/valid"])
    return dict(x=z["x"], ncat=int(z["ncat"]), cut=int(z["cut"]), cases=cases)
