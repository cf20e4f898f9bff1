// common.cuh — shared device/host helpers for libb200agg (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200agg.h"

namespace b200 {

// ---- error plumbing ----------------------------------------------------------------------------
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define B200_CUDA(expr)                                                                                                        \
    do {                                                                                                                       \
        cudaError_t e__ = (expr);                                                                                              \
        if (e__ != cudaSuccess)                                                                                                \
            return ::b200::cuda_fail(e__, #expr, __FILE__, __LINE__);                                                          \
    } while (0)

#define B200_CHECK(expr)                                                                                                       \
    do {                                                                                                                       \
        int rc__ = (expr);                                                                                                     \
        if (rc__ != B200_OK)                                                                                                   \
            return rc__;                                                                                                       \
    } while (0)

// ---- dtype tables ------------------------------------------------------------------------------
__host__ __device__ inline int dtype_size(int dt) {
    switch (dt) {
    case B200_F64:
    case B200_I64:
    case B200_U64: return 8;
    case B200_F32:
    case B200_I32:
    case B200_U32: return 4;
    case B200_I16:
    case B200_U16: return 2;
    default: return 1;
    }
}
__host__ __device__ inline bool dtype_is_float(int dt) { return dt == B200_F64 || dt == B200_F32; }
__host__ __device__ inline bool dtype_is_signed(int dt) { return dt == B200_I64 || dt == B200_I32 || dt == B200_I16 || dt == B200_I8; }
// upcast<T> of the reference (src/agg_sum.cpp:6-62): bool counts as signed
__host__ __device__ inline int dtype_upcast(int dt) {
    if (dtype_is_float(dt))
        return B200_F64;
    if (dtype_is_signed(dt) || dt == B200_BOOL)
        return B200_I64;
    return B200_U64;
}
// device cell type for min/max grids: 8/16-bit integers are held as 32-bit (no narrow atomics); widened back on read
__host__ __device__ inline int dtype_minmax_cell(int dt) {
    switch (dt) {
    case B200_I16:
    case B200_I8: return B200_I32;
    case B200_U16:
    case B200_U8:
    case B200_BOOL: return B200_U32;
    default: return dt;
    }
}

// ---- device-side context objects ---------------------------------------------------------------
struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t h2d_done = nullptr;
    void *stage = nullptr; // device staging arena for host chunks
    size_t stage_cap = 0;
    void *pinned = nullptr; // small pinned scratch (results of reductions)
    // host-chunk ingestion: a ring of kBounce page-locked pieces of kBouncePiece bytes.  The calling thread memcpy's a host column
    // piece by piece into the ring and every piece travels to the arena with its own asynchronous copy, so the call returns without
    // waiting for the device (the caller's buffer is only valid during the call, vaex/cpu.py:708-710).  The ring is small on
    // purpose (16 MB a slot whatever the chunk size): the pieces stay in the host's last-level cache between the memcpy that writes
    // them and the DMA that reads them, and no chunk-sized page-locked allocation is ever made.
    static constexpr int kBounceMax = 16;
    void *bounce[kBounceMax] = {};
    size_t bounce_cap[kBounceMax] = {};
    cudaEvent_t bounce_done[kBounceMax] = {};
    unsigned bounce_next = 0;
    // wall-clock nanoseconds of the host-chunk path on this slot (b200_ctx_host_stats): waiting for a ring piece, memcpy into it,
    // enqueueing its copy, the whole of b200_bin; pieces and calls
    uint64_t host_ns[4] = {0, 0, 0, 0}, host_pieces = 0, host_calls = 0;
    void *dscratch = nullptr;
    void *scratch = nullptr; // partition scratch (ringcount pool + list tables, tilesort buckets)
    size_t scratch_cap = 0;
    // the last ringcount batch on this slot, for b200_ctx_path_stats (device pointers into `scratch`)
    const unsigned *ring_len = nullptr, *ring_ctl = nullptr;
    size_t ring_lists = 0;
    uint64_t ring_rows = 0, ring_memset_bytes = 0, ring_chunk_entries = 0;
    std::mutex mu;
};

} // namespace b200

struct b200_ctx {
    int device = 0;
    int nslots = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    std::vector<b200::Slot *> slots;
    // Grid cache: an aggregation pass creates its aggregators and destroys them when the result has been read (vaex builds a task
    // part per pass), and cudaMalloc / cudaFree synchronise the device and take the driver's allocation lock — measured at up to
    // 45 ms a call while 16-32 feeder threads are enqueueing copies (profiles/r02_e2e_probe.txt).  Released grids are kept by exact
    // size (bounded) and handed to the next pass.
    std::mutex cache_mu;
    std::multimap<size_t, void *> cache;
    size_t cache_bytes = 0;
};

struct b200_agg {
    b200_ctx *ctx = nullptr;
    int op = 0, dtype = 0, dtype2 = 0, byteswap = 0;
    uint32_t moment = 0;
    uint64_t cells = 0;
    int cell_dtype = 0;     // device cell type of `grid`
    void *grid = nullptr;   // cells * dtype_size(cell_dtype)
    void *state = nullptr;  // FIRST/LAST: cells * 16 B {u64 order key, u64 global row}
    void *order = nullptr;  // FIRST/LAST: cells * dtype_size(dtype2) raw order values
    uint8_t *cell_masked = nullptr; // FIRST/LAST
    cudaEvent_t chain = nullptr;    // FIRST/LAST: completion of the previous select+deposit pair on this grid (any slot)
    std::mutex chain_mu;
    // NUNIQUE: `grid` holds three planes of `cells` u64 (distinct pairs, NaN rows, null rows); the distinct (cell, value) pairs
    // live in one open-addressing table of 16-byte slots
    unsigned long long *ntable = nullptr;
    uint64_t ncap = 0;                     // slots (power of two)
    unsigned long long *ntotal = nullptr;  // device counter: pairs in the table
    uint64_t npairs = 0;                   // host copy, refreshed after every launch
    std::mutex nmu;                        // growth needs the table to itself
    // LIST (list.cu): one record per row {cell * 4 + category, value bits}, appended per call, sorted when the result is asked for
    unsigned long long *list_keys = nullptr, *list_vals = nullptr;
    unsigned *list_counts = nullptr;       // after finish: exclusive offsets per cell (+ the total)
    uint64_t list_n = 0, list_cap = 0, list_total = 0;
    bool list_sorted = false;
    // LIST_STRING (list.cu): the records above with key = cell and payload = arrival index (bit 63: null string); every call's bytes
    // are appended to one device pool, record r's bytes start at str_start[r] (its length: str_start[r + 1] - str_start[r])
    unsigned char *str_pool = nullptr;
    uint64_t str_pool_n = 0, str_pool_cap = 0;
    unsigned long long *str_start = nullptr; // list_cap + 1 entries
    // after finish: int64 string offsets[list_total + 1], the gathered bytes, one null flag per element
    long long *str_off = nullptr;
    unsigned char *str_bytes = nullptr, *str_nulls = nullptr;
    uint64_t str_nbytes = 0, str_elem_cap = 0, str_bytes_cap = 0;
    bool str_ready = false; // the buffers hold the result of the last finish (cleared by a new row or a reset)
};

namespace b200 {

// staging: make `n` bytes starting at host/device pointer available on the device for this slot
struct Stager {
    b200_ctx *ctx;
    Slot *slot;
    int memspace;
    bool async_host = false; // the caller keeps its host buffers alive until b200_ctx_sync(slot): copy straight from them
    size_t used = 0;
    struct Entry {
        const void *host;
        size_t bytes;
        void *dev;
    };
    std::vector<Entry> entries;
    size_t need = 0;
    // two-phase: plan() every column, then commit() allocates once and issues the copies
    void plan(const void *p, size_t bytes);
    int commit();
    const void *dev(const void *p) const;
};

int slot_reserve(b200_ctx *ctx, Slot *s, size_t bytes);
// grid cache of the context (api.cu): cudaMalloc on a miss; a released block must not be referenced by work in flight
cudaError_t ctx_alloc(b200_ctx *ctx, void **out, size_t bytes);
void ctx_release(b200_ctx *ctx, void *p, size_t bytes);
bool is_device_pointer(const void *p);

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

} // namespace b200
