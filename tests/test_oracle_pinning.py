"""Pin the oracle (oracle/binstats_oracle.c) — CPU only — against the golden vectors generated from the compiled, unmodified
reference (tests/golden/): known-answer and fixed cases stored with their inputs, and random / quirk cases whose inputs
tests/helpers.py rebuilds from a seed (tests/golden/pinning_golden.npz).
The oracle is the checker of every GPU parity test, so it has to be right first."""
import numpy as np
import pytest

import golden_util
from helpers import (CHUNK_LOOP_THREADS, MINMAX_RANDOM_DTYPES, chunk_loop_case, first_mask_quirk_case, minmax_random_columns, random_binby_case,
                     same)

GOLD = golden_util.load()
BINBY = sorted(k for k in GOLD if not k.startswith(("set_", "hash64")))
SETS = sorted(k for k in GOLD if k.startswith("set_"))


@pytest.mark.parametrize("name", BINBY)
def test_oracle_matches_golden_binby(name, oracle):
    binners, aggs, n, expected = golden_util.binby_case(GOLD[name])
    got = oracle.binby(binners, aggs, n)
    for a, w, g in zip(aggs, expected, got):
        assert same(w, g), (name, a["op"])


def test_golden_kats_are_the_reference_test_vectors():
    # /root/reference/tests/agg_test.py:150-158 and :171-180
    assert GOLD["kat_count_1d"]["a0_result"].tolist() == [0, 2, 1, 1, 0, 0, 1, 1]
    assert GOLD["kat_count_1d_ordinal"]["a0_result"].tolist() == [1, 1, 0, 0, 1, 3, 0]


@pytest.mark.parametrize("name", SETS)
def test_oracle_matches_golden_sets(name, oracle):
    c = GOLD[name]
    dtype, nmaps = name.split("_")[1], int(name.split("_")[2])
    s = oracle.OrderedSet(dtype, nmaps)
    vals, mi = s.update(c["keys"], c["mask"], 0, True)
    assert np.array_equal(vals, c["values"]) and np.array_equal(mi, c["map_index"])
    assert np.array_equal(s.key_array(), c["key_array"], equal_nan=True)
    assert s.offsets() == c["offsets"].tolist()
    mo = s.map_ordinal(c["keys"])
    assert mo.dtype == c["map_ordinal"].dtype and np.array_equal(mo, c["map_ordinal"])
    assert [s.null_index, s.nan_index, s.null_count, s.nan_count] == c["null_nan"].tolist()


def test_hash64_golden(oracle):
    for i, o in zip(GOLD["hash64"]["in"], GOLD["hash64"]["out"]):
        assert oracle.hash64(int(i)) == int(o)
    assert oracle.hash64(1) == 6238072747940578789  # SURVEY.md 8c pin


# ---- the compiled reference's answers on the cases of tests/helpers.py (tests/golden/pinning_golden.npz) -------------------------
PINNED = golden_util.load_pinning()


@pytest.mark.parametrize("seed", range(12))
def test_oracle_matches_compiled_reference_random(seed, oracle):
    binners, aggs, n = random_binby_case(seed)
    want = golden_util.pinned_results(PINNED[f"random_{seed}"])
    got = oracle.binby(binners, aggs, n)
    assert len(want) == len(aggs)
    for a, w, g in zip(aggs, want, got):
        assert same(w, g), (a["op"], None if a["data"] is None else a["data"].dtype)


def test_oracle_first_mask_quirk_matches_reference(oracle):
    """AggFirst indexes its mask inside the 1024-row block without the block offset (src/agg_first.cpp:131);
    the oracle restates that, so both agree even past 1024 rows."""
    b, a, n = first_mask_quirk_case()
    want = golden_util.pinned_results(PINNED["first_mask_quirk"])
    assert len(want) == 2
    for w, g in zip(want, oracle.binby(b, a, n)):
        assert same(w, g)


@pytest.mark.parametrize("nthreads", CHUNK_LOOP_THREADS)
def test_reference_chunk_loop_is_thread_invariant_for_counts(nthreads, oracle):
    """the reference's executor loop (50k-row chunks over `nthreads` threads, per-thread grids folded in get_result) gives the
    counts of one sequential pass"""
    b, a, n = chunk_loop_case()
    want = oracle.binby(b, a, n)[0]
    got = golden_util.pinned_results(PINNED[f"chunk_loop_{nthreads}"])[0]
    assert int(got.sum()) == n
    assert np.array_equal(want, got)


# ---- limits pre-pass (df.minmax): SURVEY.md section 8f row 1 ------------------------------------------------------------------
MINMAX = golden_util.load_minmax()


@pytest.mark.parametrize("name", sorted(MINMAX))
def test_oracle_minmax_matches_golden(name, oracle):
    """oracle.minmax (orc_minmax) against vaexfast.statisticNd OP_MIN_MAX of the compiled reference: all 11 dtypes, masked,
    byte-swapped, NaN / inf, integers beyond 2^24 / 2^53 (rounded by the reference's float casts), empty and all-NaN columns."""
    data, raw, result = MINMAX[name]
    assert np.array_equal(oracle.minmax(data, raw=True), raw, equal_nan=True)
    got = oracle.minmax(data)
    assert got.dtype == result.dtype and np.array_equal(got, result, equal_nan=True)


def test_minmax_float_cast_quirk_is_in_the_golden_vectors():
    # int32 max - 1 = 2147483646 is not a float32: the reference reports 2147483648.0 in its grid (vaex/cpu.py:519-531)
    _, raw, _ = MINMAX["int32"]
    assert raw[1] == 2147483648.0
    _, raw, _ = MINMAX["int64"]
    assert raw[1] == 9223372036854775808.0  # int64 goes through float64


@pytest.mark.parametrize("seed", range(6))
def test_oracle_minmax_matches_compiled_reference_random(seed, oracle):
    cols = minmax_random_columns(seed)
    want = PINNED[f"minmax_{seed}"]["raw"]
    assert len(want) == len(cols) == 2 * len(MINMAX_RANDOM_DTYPES)
    for (dt, col), w in zip(cols, want):
        assert np.array_equal(oracle.minmax(col, raw=True), w, equal_nan=True), dt


# ---- string key sets (SURVEY.md section 8f row 3) ----------------------------------------------------------------------------------
STRINGS = golden_util.load_strings()


def test_string_hash_known_answers(oracle):
    """std::hash<string_view> of the reference build = libstdc++'s 64-bit Murmur-2 (src/hash.hpp:59-86)"""
    c = STRINGS["strhash"]
    keys = [bytes(c["bytes"][c["offsets"][i]:c["offsets"][i + 1]]) for i in range(len(c["offsets"]) - 1)]
    assert [oracle.string_hash(k) for k in keys] == [int(h) for h in c["hash"]]


@pytest.mark.parametrize("name", sorted(k for k in STRINGS if k.startswith("strset_")))
def test_oracle_string_set_matches_golden(name, oracle):
    c = STRINGS[name]
    s = oracle.StringOrderedSet(int(name.split("_")[1]))
    for k in range(int(c["ncalls"])):
        strs = golden_util.unpack_strings(c[f"c{k}_offsets"], c[f"c{k}_bytes"], c[f"c{k}_mask"])
        vals, mi = s.update(strs, 0, True)
        assert np.array_equal(vals, c[f"c{k}_values"]) and np.array_equal(mi, c[f"c{k}_map_index"])
    assert s.keys() == golden_util.unpack_strings(c["key_offsets"], c["key_bytes"], c["key_nulls"])
    assert s.offsets() == c["shard_offsets"].tolist()
    probe = golden_util.unpack_strings(c["probe_offsets"], c["probe_bytes"], c["probe_mask"])
    assert np.array_equal(s.map_ordinal(probe), c["probe_ordinals"])
    assert [len(s), s.null_count, s.null_index] == c["info"].tolist()


def test_agg_list_restatement_matches_the_compiled_reference_vectors():
    """oracle.agg_list (src/agg_list.cpp restated, incl. the mask-without-block-offset quirk) against the vectors the compiled
    reference's AggList_<dtype>_int64 produced (tests/golden/make_golden_agglist.py): 5 dtypes x plain / masked x dropnan x dropnull,
    fed in two calls of 1777 and 2223 rows (so the 1024-row blocks and the call boundary both matter)."""
    import golden_util
    from oracle import oracle as O
    g = golden_util.load_agglist()
    x, n = g["x"], len(g["x"])
    cells = O.flat_indices([O.ordinal(x, g["ncat"], 0)], n)[0].astype(np.int64)
    assert len(g["cases"]) == 40
    for name, c in g["cases"].items():
        off, vals, _, _ = O.agg_list(cells, c["v"], c["valid"] if c["masked"] else None, len(c["offsets"]) - 1, c["dropnan"], c["dropnull"],
                                     calls=[(0, g["cut"]), (g["cut"], n)])
        assert np.array_equal(off, c["offsets"]), name
        assert np.array_equal(vals, c["values"], equal_nan=True), name
