"""AggList_string_int64 restated in plain Python (TEST INFRASTRUCTURE ONLY; the numeric list's restatement is oracle.agg_list).

Pinned against the compiled reference by tests/golden/agglist_string_golden.npz (tests/golden/make_golden_agglist_string.py)."""
import numpy as np


def agg_list_string(cells, offsets, data, nulls=None, ncells=None, dropnull=False):
    """AggListString (src/agg_list.cpp:183-197 aggregate, :141-182 get_result) restated.

    Per cell of the flat grid, the rows' strings in arrival order (:191-192 `grid_data[i].push(string_sequence->view(j + offset))`).
    A null string becomes a null element at its arrival position, or nothing with dropnull (:193-194 `push_null()`). It does not go
    to the tail of the list, which is where the numeric AggListPrimitive puts nulls. null_count is never incremented (:137, :157),
    so it adds nothing to the offsets. dropnan is stored and never read. REFERENCE QUIRK, kept: aggregate() never reads the data mask
    (AggBaseString::set_data_mask only stores it, src/agg_base.hpp:192-198), so this takes none: a selection filters nothing.

    `cells`: flat cell of every row, rows in bin() call order; `offsets` int64[n + 1] (may start past 0) / `data` uint8 / `nulls`
    uint8 (1 = null) or None: the strings in the arrow large_string layout.  Returns (list offsets int64[ncells + 1], string
    offsets int64[nelem + 1], bytes uint8, null flags uint8[nelem]): the buffers of the large_list<large_string> the reference
    hands to vaex.arrow.convert.list_from_arrays (:179-181)."""
    cells = np.asarray(cells, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    data = np.asarray(data, dtype=np.uint8)
    ncells = int(cells.max()) + 1 if ncells is None else int(ncells)
    lists = [[] for _ in range(ncells)]
    for j, c in enumerate(cells.tolist()):
        if nulls is not None and nulls[j]:
            if not dropnull:
                lists[c].append(None)
        else:
            lists[c].append(data[offsets[j]:offsets[j + 1]].tobytes())
    list_offsets = np.zeros(ncells + 1, np.int64)
    list_offsets[1:] = np.cumsum([len(x) for x in lists])
    flat = [s for x in lists for s in x]
    str_offsets = np.zeros(len(flat) + 1, np.int64)
    str_offsets[1:] = np.cumsum([0 if s is None else len(s) for s in flat])
    out = np.frombuffer(b"".join(s for s in flat if s is not None), np.uint8).copy()
    return list_offsets, str_offsets, out, np.array([s is None for s in flat], np.uint8)
