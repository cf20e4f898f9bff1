"""AggList_string_int64 on the device (csrc/list.cu): the compiled reference's answers (tests/golden/agglist_string_golden.npz),
random cases against the plain-Python restatement (oracle/oracle_strlist.py), and the groupby / Frame paths that reach it."""
import numpy as np
import pytest

import golden_strlist

pytestmark = pytest.mark.gpu

GOLDEN = golden_strlist.load()
CASES = [(name, case) for name in GOLDEN for case in sorted(GOLDEN[name]["cases"])]


def _large_string(offsets, data, nulls):
    import pyarrow as pa
    validity = pa.py_buffer(np.packbits(nulls == 0, bitorder="little")) if nulls is not None and nulls.any() else None
    n = len(offsets) - 1
    return pa.Array.from_buffers(pa.large_string(), n, [validity, pa.py_buffer(offsets), pa.py_buffer(data)],
                                 null_count=int(nulls.sum()) if validity is not None else 0)


def _check(got, want):
    for field, g, w in zip(golden_strlist.FIELDS, got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w), field


@pytest.mark.parametrize("name,case", CASES, ids=[f"{n}-{c}" for n, c in CASES])
def test_golden_vectors_bit_identical(name, case):
    import pyarrow as pa
    from vaex_b200 import superagg
    s, c = GOLDEN[name], GOLDEN[name]["cases"][case]
    strings = _large_string(s["offsets"], s["bytes"], s["nulls"])
    b = golden_strlist.device_binner(name)
    g = superagg.Grid([b])
    a = superagg.AggList_string_int64(g, 1, 1, c["dropnan"], c["dropnull"])
    for i1, i2 in s["calls"]:  # the reference's bin() calls; every slice but the first starts past offset 0
        b.set_data(0, np.ascontiguousarray(s["x"][i1:i2]))
        a.set_data(0, strings[i1:i2], 0)
        if c["masked"]:
            a.set_data_mask(0, np.zeros(i2 - i1, np.uint8))
        g.bin(0, [a], i2 - i1)
    _check(a.result_arrays(), c["expected"])
    res = a.get_result()
    assert res.type == pa.large_list(pa.large_string()) and len(res) == len(g)


def _random_strings(rng, n, null_rate=0.1, long_rate=0.02, long_len=6000):
    lengths = rng.integers(0, 24, n)
    lengths[rng.random(n) < 0.1] = 0
    lng = rng.random(n) < long_rate
    lengths[lng] = rng.integers(33, long_len, int(lng.sum()))
    offsets = np.zeros(n + 1, np.int64)
    offsets[1:] = np.cumsum(lengths)
    data = rng.integers(32, 127, int(offsets[-1])).astype(np.uint8)
    nulls = (rng.random(n) < null_rate).astype(np.uint8)
    return offsets, data, nulls


def _feed(strings_of_call, calls, x, binner_factory, dropnull, threads=1, selection=False):
    from vaex_b200 import superagg
    b = binner_factory()
    g = superagg.Grid([b])
    a = superagg.AggList_string_int64(g, 1, threads, False, dropnull)
    for k, (i1, i2) in enumerate(calls):
        t = k % threads
        b.set_data(t, np.ascontiguousarray(x[i1:i2]))
        a.set_data(t, strings_of_call(i1, i2), 0)
        if selection:
            a.set_data_mask(t, np.zeros(i2 - i1, np.uint8))  # a selection reaches the aggregator as its data mask: ignored
        g.bin(t, [a], i2 - i1)
    return a, g


def _oracle(x, ncat, offsets, data, nulls, dropnull):
    from oracle import oracle as O
    from oracle.oracle_strlist import agg_list_string
    cells, shapes = O.flat_indices([O.ordinal(x, ncat, 0)], len(x))
    return agg_list_string(cells, offsets, data, nulls, ncells=int(np.prod(shapes)), dropnull=dropnull)


@pytest.mark.parametrize("feed", ["arrow_sliced", "arrow_string", "host_buffers", "device_buffers", "object"])
@pytest.mark.parametrize("threads", [1, 3])
@pytest.mark.parametrize("dropnull", [False, True])
def test_random_against_the_oracle(feed, threads, dropnull):
    import zlib

    import pyarrow as pa
    import torch
    from vaex_b200 import superagg
    rng = np.random.default_rng(zlib.crc32(f"{feed}/{threads}/{dropnull}".encode()))
    n, ncat = 20_000, 300  # most cells hold a few strings, many hold none
    x = rng.integers(-1, ncat + 1, n).astype("i8")
    x[rng.random(n) < 0.3] = 7  # one hot cell
    offsets, data, nulls = _random_strings(rng, n)
    whole = _large_string(offsets, data, nulls)
    calls = [(0, 3000), (3000, 3000), (3000, 11_111), (11_111, n)]

    def strings_of_call(i1, i2):
        if feed == "arrow_sliced":
            return whole[i1:i2]
        if feed == "arrow_string":
            return whole[i1:i2].cast(pa.string())
        if feed == "object":
            return np.array(whole[i1:i2].to_pylist(), dtype=object)
        off = offsets[i1:i2 + 1]
        if feed == "host_buffers":
            return off, data, nulls[i1:i2]
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        return dev(off), dev(data), dev(nulls[i1:i2])

    a, _ = _feed(strings_of_call, calls, x, lambda: superagg.BinnerOrdinal_int64(1, "x", ncat, 0, False, False), dropnull, threads=threads, selection=True)
    _check(a.result_arrays(), _oracle(x, ncat, offsets, data, nulls, dropnull))


def test_get_result_is_an_arrow_list_of_strings_with_nulls_in_place():
    from vaex_b200 import superagg
    x = np.array([0, 1, 0, 2, 1, 0, 5], "i8")
    b = superagg.BinnerOrdinal_int64(1, "x", 3, 0, False, False)
    g = superagg.Grid([b])
    a = superagg.AggList_string_int64(g, 1, 1)
    b.set_data(0, x)
    a.set_data(0, ["a", None, "bcd", "", "zz", None, "q"])
    g.bin(0, [a], 7)
    assert a.get_result().to_pylist() == [["a", "bcd", None], [None, "zz"], [""], ["q"], []]
    assert a.merge([]) is None and a.__sizeof__() == 0
    with pytest.raises(RuntimeError, match="only accepts 1 grid"):
        superagg.AggList_string_int64(g, 2, 1)


@pytest.mark.parametrize("combine", [False, True])
@pytest.mark.parametrize("by_col_has_missing", [False, True])
@pytest.mark.parametrize("dropmissing", [False, True])
def test_groupby_agg_list_strings(dropmissing, by_col_has_missing, combine):
    # tests/agg_test.py:663-694 (test_agg_list), both columns: groupby('id').agg({'food': list(food), 'num': list(num)})
    import pyarrow as pa
    from vaex_b200 import agg
    from vaex_b200.frame import Frame
    ids = np.ma.array([1, 2, 2, 1, 1, 3, 3], mask=[0, 0, 0, 0, 0, by_col_has_missing, by_col_has_missing], dtype="i8")
    food = pa.array(["cake", "apples", "oranges", "meat", "meat", "carrots", None])
    num = np.array([1.1, 1.2, 1.3, 1.4, np.nan, 1.6, 1.7])
    cols = dict(id=ids, food=food, num=num)
    by = "id"
    if combine:
        cols["one"] = np.zeros(7, "i4")
        by = ["id", "one"]
    out = Frame(cols).groupby(by, agg={"food": agg.list("food", dropmissing=dropmissing), "num": agg.list("num", dropnan=True)}, combine=combine, sort=True)
    assert out["food"].type == pa.large_list(pa.large_string())
    want = [["cake", "meat", "meat"], ["apples", "oranges"], ["carrots"] if dropmissing else ["carrots", None]]
    assert out["food"].to_pylist() == want
    assert out["num"].to_pylist() == [[1.1, 1.4], [1.2, 1.3], [1.6, 1.7]]
    assert out["id"].tolist() == ([1, 2, None] if by_col_has_missing else [1, 2, 3])


def test_groupby_string_key_with_string_list():
    from vaex_b200 import agg
    from vaex_b200.execution import Executor
    from vaex_b200.frame import Frame
    import pyarrow as pa
    rng = np.random.default_rng(5)
    n = 30_000
    keys = np.array(["k%d" % i for i in rng.integers(0, 50, n)], dtype=object)
    keys[rng.random(n) < 0.05] = None
    vals = np.array(["v%d" % i if i % 7 else None for i in rng.integers(0, 10_000, n)], dtype=object)
    df = Frame(dict(k=pa.array(keys), s=pa.array(vals)), executor=Executor(nthreads=1, chunk_size=7_000))
    out = df.groupby("k", agg={"s": agg.list("s")})
    got = dict(zip(out["k"].tolist(), out["s"].to_pylist()))
    want = {}
    for k, v in zip(keys.tolist(), vals.tolist()):
        want.setdefault(k, []).append(v)
    assert got == want  # one worker: arrival order == row order, nulls where they arrived


def test_frame_list_strings_through_the_task_part():
    from vaex_b200.execution import Executor
    from vaex_b200.frame import Frame
    import pyarrow as pa
    rng = np.random.default_rng(9)
    n = 50_000
    x = rng.uniform(-1, 11, n)
    offsets, data, nulls = _random_strings(rng, n)
    s = _large_string(offsets, data, nulls)
    py = s.to_pylist()
    cell = np.where(np.isnan(x), 0, np.where(x < 0, 1, np.where(x >= 10, 7, np.floor(x / 2) + 2))).astype(int)
    key = lambda v: (v is None, v or "")
    lists = Frame(dict(x=x, s=s), executor=Executor(nthreads=3, chunk_size=7_001)).list("s", binby="x", limits=[0, 10], shape=5)
    assert len(lists) == 8
    for c in range(8):
        want = [py[i] for i in np.nonzero(cell == c)[0]]
        assert sorted(lists[c].as_py(), key=key) == sorted(want, key=key)  # chunks fed concurrently: order across chunks varies
    single = Frame(dict(x=x, s=s), executor=Executor(nthreads=1, chunk_size=7_001)).list("s", binby="x", limits=[0, 10], shape=5)
    for c in range(8):
        assert single[c].as_py() == [py[i] for i in np.nonzero(cell == c)[0]]  # sequential feed: exactly row order


def _numpy_restatement(cells, ncells, offsets, data, nulls, dropnull):
    """agg_list_string vectorised (stable sort by cell), for sizes the Python loop of the oracle cannot take"""
    keep = np.ones(len(cells), bool) if not dropnull else nulls == 0
    rows = np.nonzero(keep)[0]
    order = rows[np.argsort(cells[rows], kind="stable")]
    list_offsets = np.zeros(ncells + 1, np.int64)
    list_offsets[1:] = np.cumsum(np.bincount(cells[rows], minlength=ncells))
    lens = np.where(nulls[order] != 0, 0, offsets[order + 1] - offsets[order])
    str_offsets = np.zeros(len(order) + 1, np.int64)
    str_offsets[1:] = np.cumsum(lens)
    pos = np.arange(int(str_offsets[-1]), dtype=np.int64) + np.repeat(offsets[order] - str_offsets[:-1], lens)
    return list_offsets, str_offsets, data[pos], nulls[order].astype(np.uint8)


def test_ten_million_rows_grow_the_pool_across_calls():
    from oracle import oracle as O
    from oracle.oracle_strlist import agg_list_string
    from vaex_b200 import superagg
    rng = np.random.default_rng(11)
    n, ncat = 10_000_000, 1000
    x = rng.integers(0, ncat, n).astype("i8")
    lengths = rng.integers(0, 20, n)
    offsets = np.zeros(n + 1, np.int64)
    offsets[1:] = np.cumsum(lengths)
    data = rng.integers(97, 123, int(offsets[-1])).astype(np.uint8)
    nulls = (rng.random(n) < 0.05).astype(np.uint8)
    cells = O.flat_indices([O.ordinal(x, ncat, 0)], n)[0].astype(np.int64)
    ncells = ncat + 2
    k = 3000  # the vectorised restatement is the oracle's own answer on a prefix
    small = _numpy_restatement(cells[:k], ncells, offsets[:k + 1], data, nulls[:k], False)
    _check(small, agg_list_string(cells[:k], offsets[:k + 1], data, nulls[:k], ncells=ncells))
    calls = [(i, min(i + 1_300_000, n)) for i in range(0, n, 1_300_000)]
    a, _ = _feed(lambda i1, i2: (offsets[i1:i2 + 1], data, nulls[i1:i2]), calls, x,
                 lambda: superagg.BinnerOrdinal_int64(1, "x", ncat, 0, False, False), False, threads=4)
    _check(a.result_arrays(), _numpy_restatement(cells, ncells, offsets, data, nulls, False))
