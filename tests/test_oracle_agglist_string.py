"""The plain-Python restatement of AggList_string_int64 (oracle/oracle_strlist.py) against what the compiled reference returned
(tests/golden/agglist_string_golden.npz).  No GPU needed."""
import numpy as np
import pytest

import golden_strlist

GOLDEN = golden_strlist.load()
CASES = [(name, case) for name in GOLDEN for case in sorted(GOLDEN[name]["cases"])]


@pytest.mark.parametrize("name,case", CASES, ids=[f"{n}-{c}" for n, c in CASES])
def test_restatement_reproduces_the_reference(oracle, name, case):
    from oracle.oracle_strlist import agg_list_string
    s, c = GOLDEN[name], GOLDEN[name]["cases"][case]
    cells, shapes = oracle.flat_indices([golden_strlist.oracle_binner(name, s["x"])], len(s["x"]))
    # the data mask is not an input: the reference never reads it, so the masked and plain cases must agree
    got = agg_list_string(cells, s["offsets"], s["bytes"], s["nulls"], ncells=int(np.prod(shapes)), dropnull=c["dropnull"])
    for field, g, w in zip(golden_strlist.FIELDS, got, c["expected"]):
        assert g.dtype == w.dtype and np.array_equal(g, w), field


def test_small_example_nulls_stay_in_arrival_order():
    from oracle.oracle_strlist import agg_list_string
    from vaex_b200.superutils import string_buffers
    cells = [0, 1, 0, 2, 1, 0, 3]  # ordinal binner, 3 categories: 5 cells, value 5 lands in the first edge cell
    offsets, data, nulls = string_buffers(["a", None, "bcd", "", "zz", None, "q"])
    lo, so, b, nf = agg_list_string(cells, offsets, data, nulls, ncells=5)
    assert lo.tolist() == [0, 3, 5, 6, 7, 7]
    assert nf.tolist() == [0, 0, 1, 1, 0, 0, 0]  # [a, bcd, null] [null, zz] [""] [q] []
    assert [bytes(b[so[i]:so[i + 1]]) for i in range(7)] == [b"a", b"bcd", b"", b"", b"zz", b"", b"q"]
    lo, so, b, nf = agg_list_string(cells, offsets, data, nulls, ncells=5, dropnull=True)
    assert lo.tolist() == [0, 2, 3, 4, 5, 5] and not nf.any()


def test_find_type_resolves_the_string_list_class():
    from vaex_b200 import agg, superagg
    assert agg.find_type_from_dtype(superagg, "AggList_", np.dtype("O"), np.dtype("int64")) is superagg.AggList_string_int64
    assert agg.find_type_from_dtype(superagg, "AggCount_", np.dtype("O")) is superagg.AggCount_string
    with pytest.raises(ValueError, match="AggFirst_string_int64"):
        agg.find_type_from_dtype(superagg, "AggFirst_", np.dtype("O"), np.dtype("int64"))
