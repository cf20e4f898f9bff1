// oracle/ref_strlist_shim.cpp — TEST INFRASTRUCTURE ONLY.
// glue only: registers the reference's StringSequence / StringList64 (src/superstring.hpp, unmodified, included from where it lies)
// with pybind11 under shared_ptr holders, like the reference's own `superstrings` module does (which needs pcre and is not built
// here).  pybind11 shares its type registry between the modules of one process, so the compiled reference's AggList_string_int64
// (oracle/_ref/superagg) accepts these objects in set_data and returns one from get_result.
#include "superstring.hpp"
namespace py = pybind11;

// (int64 offsets[n + 1], uint8 bytes, uint8 null mask (1 = null) or None) -> StringList64; offsets may start past 0
static std::shared_ptr<StringList64> string_list(py::array_t<int64_t> offsets, py::array_t<uint8_t> bytes, py::object mask) {
    const int64_t n = offsets.shape(0) - 1;
    const int64_t first = offsets.at(0), nbytes = offsets.at(n) - first;
    auto sl = std::make_shared<StringList64>(nbytes, n);
    std::copy(bytes.data() + first, bytes.data() + first + nbytes, (uint8_t *)sl->bytes);
    for (int64_t i = 0; i <= n; i++)
        sl->indices[i] = offsets.at(i) - first;
    if (!mask.is_none()) {
        py::array_t<uint8_t> m = mask.cast<py::array_t<uint8_t>>();
        sl->ensure_null_bitmap();
        for (int64_t i = 0; i < n; i++)
            if (m.at(i))
                sl->set_null(i);
    }
    return sl;
}

// StringList64 -> (int64 offsets[n + 1] starting at 0, uint8 bytes, uint8 null flags[n])
static py::tuple to_numpy(const StringList64 &sl) {
    const int64_t n = sl.length;
    py::array_t<int64_t> off(n + 1);
    for (int64_t i = 0; i <= n; i++)
        off.mutable_at(i) = sl.indices[i] - sl.indices[0];
    const int64_t nb = sl.indices[n] - sl.indices[0];
    py::array_t<uint8_t> by(nb);
    std::copy(sl.bytes + sl.indices[0] - sl.offset, sl.bytes + sl.indices[0] - sl.offset + nb, (char *)by.mutable_data());
    py::array_t<uint8_t> nulls(n);
    for (int64_t i = 0; i < n; i++)
        nulls.mutable_at(i) = sl.is_null(i);
    return py::make_tuple(off, by, nulls);
}

PYBIND11_MODULE(strlist_shim, m) {
    py::class_<StringSequence, std::shared_ptr<StringSequence>> seq(m, "StringSequence");
    py::class_<StringList64, std::shared_ptr<StringList64>>(m, "StringList64", seq).def("__len__", [](const StringList64 &s) { return s.length; });
    m.def("string_list", &string_list);
    m.def("to_numpy", &to_numpy);
}
