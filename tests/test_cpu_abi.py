"""CPU-side checks of the boundary: the C-ABI library loads, exports every symbol include/b200agg.h declares, the
mirror modules expose the reference's class names, and the product fails LOUDLY (no CPU fallback) without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

import golden_util
from helpers import grid_layout_binners

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200agg.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from vaex_b200 import _lib
    _lib.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 40
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert L.b200_abi_version() == 1


def test_binding_covers_header():
    """every declared entry point has a ctypes signature in the binding (so nothing is called with default int args)"""
    from vaex_b200 import _lib
    src = open(os.path.join(ROOT, "vaex_b200", "_lib.py")).read()
    bound = set(re.findall(r'"(b200_[a-z0-9_]+)":', src))
    assert set(declared_symbols()) <= bound, set(declared_symbols()) - bound


def test_hash64_known_answers():
    # superutils.hash pins verified against the compiled reference (SURVEY.md section 8c)
    from vaex_b200 import superutils
    assert superutils.hash(1) == 6238072747940578789
    assert superutils.hash(2) == 15839785061582574730


def test_mirror_class_names_match_reference():
    """every numeric Binner*/Agg* name of the compiled reference module resolves in the mirror (names stored by
    tests/golden/make_golden_pinning.py)"""
    from vaex_b200 import superagg as mine, superutils as myutils
    names = golden_util.load_pinning()["names"]
    want = [str(n) for n in names["superagg"]]
    assert len(want) > 300
    missing = [n for n in want if not hasattr(mine, n)]
    assert not missing, missing[:10]
    assert hasattr(mine, "Grid")
    sets = [str(n) for n in names["ordered_sets"]]
    assert len(sets) == 11
    assert not [n for n in sets if not hasattr(myutils, n)]


def test_string_names_resolve_and_object_names_raise():
    from vaex_b200 import superagg, superutils
    assert superagg.AggNUnique_string and superagg.AggCount_string and superutils.ordered_set_string  # round 2: string keys on the device
    with pytest.raises(AttributeError):
        superagg.AggCount_object


def test_no_cpu_fallback():
    """without a GPU the product raises instead of computing on the host"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from vaex_b200 import superagg, superutils
    b = superagg.BinnerScalar_float64(1, "x", 0, 1, 4)
    g = superagg.Grid([b])
    assert len(g) == 7 and g.shapes == [7] and g.strides == [1]
    with pytest.raises(RuntimeError):
        superagg.AggCount_float64(g, 1, 1)
    with pytest.raises(RuntimeError):
        superutils.ordered_set_int64(1)


def test_grid_layout_matches_reference():
    """the mirror's Grid over grid_layout_binners has the shapes, strides and length the compiled reference's Grid has"""
    from vaex_b200 import superagg as mine
    want = golden_util.load_pinning()["grid_layout"]
    mb = grid_layout_binners(mine)
    mg = mine.Grid(mb)
    assert want["shapes"].tolist() == mg.shapes and want["strides"].tolist() == mg.strides and int(want["length"]) == len(mg)
    assert want["binner_lengths"].tolist() == [len(b) for b in mb]


def test_binner_errors_match_reference():
    from vaex_b200 import superagg
    b = superagg.BinnerScalar_float64(1, "x", 0, 1, 4)
    with pytest.raises(RuntimeError, match="Expected a 1d array"):
        b.set_data(0, np.zeros((2, 2)))
    with pytest.raises(RuntimeError, match="Itemsize of data and binner are not equal"):
        b.set_data(0, np.zeros(4, "f4"))
