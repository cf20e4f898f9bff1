// list.cu — AggList_<dtype>: per cell the list of the rows' values (SURVEY.md section 8f row 4).
//
// Reference: AggListPrimitive (src/agg_list.cpp:5-127): `grids` must be 1; aggregate() appends every valid, non-NaN value to its
// cell's std::vector, counts NaN values (unless dropnan) and null rows (data mask == 0, unless dropnull) per cell; get_result()
// returns offsets[cells + 1] + flat values: a cell's values in arrival order, then one NaN per counted NaN, then one (unwritten)
// slot per counted null — handed to vaex.arrow.convert.list_from_arrays.
// Device design: nothing cell-shaped is kept.  Every b200_bin call appends one record per row — key = cell * 4 + category (0 value,
// 1 NaN, 2 null; skipped rows get the all-ones key), payload = the value's bits — to a growing pair of device arrays, at positions
// reserved per call, so arrival order is (call, row) order.  Finishing = one stable LSD radix sort of the records by key (radix.cuh,
// only the bytes that vary) + a per-cell count + a scan: the sorted payloads ARE the flat values.
#include <algorithm>

#include "binby.cuh"
#include "binby_index.cuh"
#include "radix.cuh"
#include "scan.cuh"

namespace b200 {

struct ListParams {
    int nb;
    long long nrows;
    DevBinner b[B200_MAX_BINNERS];
    int dtype, isz, byteswap, dropnan, dropnull;
    const void *data;
    const uint8_t *mask; // aggregator convention: 1 = use the row, 0 = null row
    unsigned long long *keys, *vals;
    unsigned long long base;
    unsigned long long skip_key; // cells * 4: sorts behind every real record, costs no extra radix pass
};

namespace {

template <bool VEC>
__global__ void __launch_bounds__(256) k_list_append(const __grid_constant__ ListParams p) {
    const long long step = (long long)gridDim.x * 256 * 4;
    for (long long base = ((long long)blockIdx.x * 256 + threadIdx.x) * 4; base < p.nrows; base += step) {
        const long long left = p.nrows - base;
        const int nv = left < 4 ? (int)left : 4;
        unsigned long long idx[4];
        binby_indices<VEC>(p.b, p.nb, base, nv, idx);
        uint64_t r[4] = {0, 0, 0, 0};
        unsigned m[4] = {1, 1, 1, 1};
        load4_raw<VEC>(p.data, p.isz, base, nv, r);
        // REFERENCE QUIRK, kept (golden vectors from the compiled reference pin it): AggListPrimitive::aggregate runs per 1024-row
        // block of a bin() call with the block offset applied to the data but NOT to the mask (src/agg_list.cpp:96-97), so row r of
        // a call is judged by mask[r % 1024] — the same slip as AggFirst (src/agg_first.cpp:131).  base is a multiple of 4.
        if (p.mask)
            load4_mask<VEC>(p.mask, base & 1023, nv, m);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j >= nv)
                break;
            const uint64_t raw = p.byteswap ? bswap(r[j], p.isz) : r[j];
            unsigned long long key;
            if (m[j] == 1) {
                if (!raw_isnan(p.dtype, raw))
                    key = idx[j] * 4 + 0;
                else
                    key = p.dropnan ? p.skip_key : idx[j] * 4 + 1;
            } else {
                key = (m[j] == 0 && !p.dropnull) ? idx[j] * 4 + 2 : p.skip_key;
            }
            p.keys[p.base + base + j] = key;
            p.vals[p.base + base + j] = raw;
        }
    }
}

__global__ void k_list_count(const unsigned long long *keys, unsigned long long n, unsigned *counts, unsigned long long cells) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long k = keys[i];
        if ((k >> 2) < cells)
            atomicAdd(counts + (k >> 2), 1u);
    }
}

__global__ void k_list_values(const unsigned long long *keys, const unsigned long long *vals, unsigned long long total, int dtype, int isz, void *out) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned cat = (unsigned)(keys[i] & 3ull);
        unsigned long long v = vals[i];
        if (cat == 1) // std::numeric_limits<T>::quiet_NaN()
            v = dtype == B200_F64 ? 0x7ff8000000000000ull : 0x7fc00000ull;
        else if (cat == 2)
            v = 0; // the reference leaves these slots unwritten
        switch (isz) {
        case 8: static_cast<unsigned long long *>(out)[i] = v; break;
        case 4: static_cast<unsigned *>(out)[i] = (unsigned)v; break;
        case 2: static_cast<unsigned short *>(out)[i] = (unsigned short)v; break;
        default: static_cast<unsigned char *>(out)[i] = (unsigned char)v; break;
        }
    }
}

int nblocks_for(unsigned long long n) {
    const unsigned long long b = (n + 255) / 256;
    return (int)std::max<unsigned long long>(1, std::min<unsigned long long>(b, 148ull * 16));
}

// ---- AggList_string ------------------------------------------------------------------------------------------------------------
// Reference: AggListString (src/agg_list.cpp:122-207): aggregate() pushes every string of the call, a null string as a null element
// at its arrival position (unless dropnull), into its cell's StringList64; the data mask is never read and dropnan has no effect;
// get_result() returns offsets[cells + 1] + one StringList64 of all cells' elements.  Device design: the numeric list's records with
// key = cell (strings and nulls share it, so a stable sort keeps their arrival order) and payload = arrival index | null << 63; the
// bytes of every call are copied once into a growing pool.  Finishing = the radix sort + per-cell counts + a scan of the sorted
// elements' lengths (int64 string offsets) + one gather of the bytes into the flat output.
constexpr unsigned long long kStrNull = 1ull << 63;

struct StrListParams {
    int nb;
    long long nrows;
    DevBinner b[B200_MAX_BINNERS];
    int dropnull;
    const long long *offsets; // the call's string offsets[nrows + 1]; offsets[j] - first = byte position inside the call
    long long first;
    const uint8_t *nulls; // 1 = null string; nullable
    unsigned long long *keys, *vals, *start;
    unsigned long long base, pool_base;
    unsigned long long skip_key; // cells: behind every real record
};

template <bool VEC>
__global__ void __launch_bounds__(256) k_strlist_append(const __grid_constant__ StrListParams p) {
    const long long step = (long long)gridDim.x * 256 * 4;
    for (long long base = ((long long)blockIdx.x * 256 + threadIdx.x) * 4; base < p.nrows; base += step) {
        const long long left = p.nrows - base;
        const int nv = left < 4 ? (int)left : 4;
        unsigned long long idx[4];
        binby_indices<VEC>(p.b, p.nb, base, nv, idx);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j >= nv)
                break;
            const long long row = base + j;
            const bool null = p.nulls && p.nulls[row];
            const unsigned long long rec = p.base + (unsigned long long)row;
            p.keys[rec] = (null && p.dropnull) ? p.skip_key : idx[j];
            p.vals[rec] = rec | (null ? kStrNull : 0ull);
            p.start[rec] = p.pool_base + (unsigned long long)(p.offsets[row] - p.first);
        }
    }
}

// the keys are sorted: a warp's 32 keys are mostly one cell, so one lane adds for all lanes of its cell (with few cells, every
// resident warp would otherwise hit the same handful of counters)
__global__ void k_strlist_count(const unsigned long long *keys, unsigned long long n, unsigned *counts, unsigned long long cells) {
    const unsigned lane = threadIdx.x & 31;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long base = (unsigned long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {
        const unsigned long long i = base + lane;
        const unsigned long long k = i < n ? keys[i] : cells;
        const unsigned m = __match_any_sync(0xffffffffu, k);
        if (k < cells && lane == (unsigned)(__ffs(m) - 1))
            atomicAdd(counts + k, (unsigned)__popc(m));
    }
}

// string offsets of the sorted elements: tiles of kStrTile elements; pass 1 sums every tile's lengths, a one-CTA scan turns the sums
// into tile bases, pass 2 scans inside the tile (256 consecutive elements per round, so every load is coalesced)
constexpr int kStrTileRounds = 8;
constexpr unsigned long long kStrTile = 256ull * kStrTileRounds;

__device__ __forceinline__ unsigned long long strlist_len(const unsigned long long *vals, const unsigned long long *start, unsigned long long i) {
    const unsigned long long v = vals[i];
    if (v & kStrNull)
        return 0; // StringList::push_null: a null element has no bytes
    const unsigned long long r = v & ~kStrNull;
    return start[r + 1] - start[r];
}

__global__ void __launch_bounds__(256) k_strlist_tile_sums(const unsigned long long *vals, const unsigned long long *start, unsigned long long total,
                                                           unsigned long long *tile_sums) {
    __shared__ unsigned long long warp_sum[8];
    const unsigned long long t0 = (unsigned long long)blockIdx.x * kStrTile;
    unsigned long long s = 0;
    for (int k = 0; k < kStrTileRounds; k++) {
        const unsigned long long i = t0 + (unsigned long long)k * 256 + threadIdx.x;
        if (i < total)
            s += strlist_len(vals, start, i);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1)
        s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0)
        warp_sum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long b = 0;
        for (int w = 0; w < 8; w++)
            b += warp_sum[w];
        tile_sums[blockIdx.x] = b;
    }
}

__global__ void __launch_bounds__(256) k_strlist_offsets(const unsigned long long *vals, const unsigned long long *start, unsigned long long total,
                                                         const unsigned long long *tile_base, long long *str_off, unsigned char *nulls) {
    __shared__ unsigned long long warp_incl[8];
    __shared__ unsigned long long carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0)
        carry = tile_base[blockIdx.x];
    __syncthreads();
    const unsigned long long t0 = (unsigned long long)blockIdx.x * kStrTile;
    for (int k = 0; k < kStrTileRounds; k++) {
        const unsigned long long i = t0 + (unsigned long long)k * 256 + threadIdx.x;
        if (t0 + (unsigned long long)k * 256 >= total)
            break; // uniform
        unsigned long long len = 0;
        if (i < total) {
            len = strlist_len(vals, start, i);
            nulls[i] = (vals[i] & kStrNull) ? 1 : 0;
        }
        unsigned long long x = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o)
                x += y;
        }
        if (lane == 31)
            warp_incl[warp] = x;
        __syncthreads();
        unsigned long long before = carry;
        for (int w = 0; w < warp; w++)
            before += warp_incl[w];
        if (i < total)
            str_off[i] = (long long)(before + x - len);
        __syncthreads();
        if (threadIdx.x == 255)
            carry = before + x;
        __syncthreads();
    }
}

// copy n bytes with the whole warp: byte head up to a 16-byte aligned destination, then 16-byte stores (built from five aligned 32-bit
// loads and funnel shifts when the source is not 16-byte congruent), then a byte tail.  The pool carries 16 bytes of slack at its end
// for the word loads that reach past the last string.
__device__ __forceinline__ void warp_copy(unsigned char *dst, const unsigned char *src, unsigned long long n, int lane) {
    const unsigned long long head = min(n, (unsigned long long)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15));
    if ((unsigned long long)lane < head)
        dst[lane] = src[lane];
    dst += head, src += head, n -= head;
    const unsigned long long nvec = n / 16;
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
    if (!(reinterpret_cast<uintptr_t>(src) & 15)) {
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
        for (unsigned long long k = lane; k < nvec; k += 32)
            d4[k] = s4[k];
    } else {
        const unsigned sh = (unsigned)(reinterpret_cast<uintptr_t>(src) & 3) * 8;
        const unsigned *w = reinterpret_cast<const unsigned *>(reinterpret_cast<uintptr_t>(src) & ~uintptr_t(3));
        for (unsigned long long k = lane; k < nvec; k += 32) {
            const unsigned *q = w + k * 4;
            const unsigned w0 = q[0], w1 = q[1], w2 = q[2], w3 = q[3], w4 = q[4];
            d4[k] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
        }
    }
    for (unsigned long long k = nvec * 16 + lane; k < n; k += 32)
        dst[k] = src[k];
}

// the byte gather: a warp takes 32 consecutive elements; a short string is copied by its own lane, every long one by the whole warp
constexpr unsigned long long kStrShort = 32;

__global__ void __launch_bounds__(256) k_strlist_gather(const unsigned long long *vals, const unsigned long long *start, const long long *str_off,
                                                        const unsigned char *pool, unsigned long long total, unsigned char *out) {
    const int lane = threadIdx.x & 31;
    const unsigned long long nwarps = (unsigned long long)gridDim.x * 8;
    for (unsigned long long g = (unsigned long long)blockIdx.x * 8 + (threadIdx.x >> 5); g * 32 < total; g += nwarps) {
        const unsigned long long i = g * 32 + lane;
        unsigned long long len = 0, src = 0, dst = 0;
        if (i < total) {
            dst = (unsigned long long)str_off[i];
            len = (unsigned long long)str_off[i + 1] - dst;
            if (len)
                src = start[vals[i] & ~kStrNull];
        }
        const bool lng = len > kStrShort;
        if (!lng)
            for (unsigned long long c = 0; c < len; c++)
                out[dst + c] = pool[src + c];
        unsigned m = __ballot_sync(0xffffffffu, lng);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const unsigned long long s = __shfl_sync(0xffffffffu, src, l), d = __shfl_sync(0xffffffffu, dst, l), n = __shfl_sync(0xffffffffu, len, l);
            warp_copy(out + d, pool + s, n, lane);
        }
    }
}

// grow a device array under the aggregator's lock: every slot's work is finished first (cudaDeviceSynchronize), the kept prefix copied
template <class T>
int grow_device(T **p, uint64_t keep, uint64_t cap) {
    T *np = nullptr;
    B200_CUDA(cudaMalloc(&np, cap * sizeof(T)));
    if (keep)
        B200_CUDA(cudaMemcpy(np, *p, keep * sizeof(T), cudaMemcpyDeviceToDevice));
    cudaFree(*p);
    *p = np;
    return B200_OK;
}

// stable LSD radix sort of the aggregator's records by key (keys <= maxkey), in place; only the bytes that can differ are sorted on
int sort_records(b200_agg *a, cudaStream_t st, unsigned long long maxkey) {
    const uint64_t n = a->list_n;
    const unsigned nblk = radix_blocks(n), tiles = radix_tiles(n);
    unsigned long long *kb = nullptr, *vb = nullptr;
    unsigned *hist = nullptr;
    struct Free {
        void *p[3];
        ~Free() {
            for (void *q : p)
                cudaFree(q);
        }
    } scratch{};
    B200_CUDA(cudaMalloc(&kb, n * 8));
    scratch.p[0] = kb;
    B200_CUDA(cudaMalloc(&vb, n * 8));
    scratch.p[1] = vb;
    B200_CUDA(cudaMalloc(&hist, (size_t)256 * nblk * 4));
    scratch.p[2] = hist;
    unsigned long long *kin = a->list_keys, *vin = a->list_vals, *kout = kb, *vout = vb;
    for (int shift = 0; shift < 64 && (maxkey >> shift); shift += 8) {
        k_radix_hist<<<nblk, kRadixThreads, 0, st>>>(kin, vin, n, shift, 0, hist, nblk, tiles);
        k_scan_u32<<<1, 1024, 0, st>>>(hist, 256ull * nblk);
        k_radix_scatter<<<nblk, kRadixThreads, 0, st>>>(kin, vin, kout, vout, n, shift, 0, hist, nblk, tiles);
        B200_CUDA(cudaGetLastError());
        std::swap(kin, kout);
        std::swap(vin, vout);
    }
    B200_CUDA(cudaStreamSynchronize(st));
    if (kin != a->list_keys) { // an odd number of passes: the sorted records sit in the scratch arrays, which have n entries
        B200_CUDA(cudaMemcpy(a->list_keys, kin, n * 8, cudaMemcpyDeviceToDevice));
        B200_CUDA(cudaMemcpy(a->list_vals, vin, n * 8, cudaMemcpyDeviceToDevice));
    }
    return B200_OK;
}

} // namespace

// one b200_bin call: reserve nrows records, append (api.cu calls this for B200_AGG_LIST aggregators)
int bin_list(b200_ctx *ctx, Slot *sl, b200_agg *a, const DevBinner *db, int nbinners, const void *data, const uint8_t *mask, int64_t nrows, bool vec) {
    unsigned long long base;
    {
        std::lock_guard<std::mutex> g(a->nmu);
        if (a->list_n + (uint64_t)nrows > a->list_cap) { // grow: other slots may be appending into the old arrays
            B200_CUDA(cudaDeviceSynchronize());
            const uint64_t cap = std::max<uint64_t>((a->list_n + (uint64_t)nrows) * 2, 1u << 16);
            unsigned long long *nk = nullptr, *nv = nullptr;
            B200_CUDA(cudaMalloc(&nk, cap * 8));
            B200_CUDA(cudaMalloc(&nv, cap * 8));
            if (a->list_n) {
                B200_CUDA(cudaMemcpy(nk, a->list_keys, a->list_n * 8, cudaMemcpyDeviceToDevice));
                B200_CUDA(cudaMemcpy(nv, a->list_vals, a->list_n * 8, cudaMemcpyDeviceToDevice));
            }
            cudaFree(a->list_keys);
            cudaFree(a->list_vals);
            a->list_keys = nk, a->list_vals = nv, a->list_cap = cap;
        }
        base = a->list_n;
        a->list_n += (uint64_t)nrows;
        a->list_sorted = false;
    }
    ListParams p;
    memset(&p, 0, sizeof p);
    p.nb = nbinners;
    p.nrows = nrows;
    memcpy(p.b, db, sizeof(DevBinner) * nbinners);
    p.dtype = a->dtype;
    p.isz = dtype_size(a->dtype);
    p.byteswap = a->byteswap && p.isz > 1;
    p.dropnan = (a->moment & 1) != 0; // AggList_<T>(grid, grids, threads, dropnan, dropnull): carried in `moment` like NUNIQUE's flags
    p.dropnull = (a->moment & 2) != 0;
    p.data = data;
    p.mask = mask;
    p.keys = a->list_keys;
    p.vals = a->list_vals;
    p.base = base;
    p.skip_key = a->cells * 4;
    const bool v = vec && !(reinterpret_cast<uintptr_t>(data) & 15) && !(reinterpret_cast<uintptr_t>(mask) & 15);
    const int blocks = nblocks_for(((unsigned long long)nrows + 3) / 4);
    if (v)
        k_list_append<true><<<blocks, 256, 0, sl->stream>>>(p);
    else
        k_list_append<false><<<blocks, 256, 0, sl->stream>>>(p);
    B200_CUDA(cudaGetLastError());
    (void)ctx;
    return B200_OK;
}

// one b200_bin call of a B200_AGG_LIST_STRING aggregator: `offsets` / `bytes` / `nulls` are the call's staged string columns (device
// pointers; bytes holds the call's nbytes bytes, offsets[j] - first indexes it).  The records and the byte range are reserved, the
// bytes copied into the pool and the records written while the aggregator's lock is held, so a growth on another slot (which waits
// for the whole device) can never free arrays that a launched-but-unfinished call still writes.
int bin_list_string(Slot *sl, b200_agg *a, const DevBinner *db, int nbinners, const long long *offsets, const unsigned char *bytes, long long first,
                    unsigned long long nbytes, const uint8_t *nulls, int64_t nrows, bool vec) {
    std::lock_guard<std::mutex> g(a->nmu);
    cudaStream_t st = sl->stream;
    if (a->list_n + (uint64_t)nrows > a->list_cap) {
        B200_CUDA(cudaDeviceSynchronize());
        const uint64_t cap = std::max<uint64_t>((a->list_n + (uint64_t)nrows) * 2, 1u << 16);
        B200_CHECK(grow_device(&a->list_keys, a->list_n, cap));
        B200_CHECK(grow_device(&a->list_vals, a->list_n, cap));
        B200_CHECK(grow_device(&a->str_start, a->list_n, cap + 1));
        a->list_cap = cap;
    }
    if (a->str_pool_n + nbytes + 16 > a->str_pool_cap) { // 16 bytes of slack behind the last string for the gather's word loads
        B200_CUDA(cudaDeviceSynchronize());
        const uint64_t cap = std::max<uint64_t>((a->str_pool_n + nbytes + 16) * 2, 1u << 20);
        B200_CHECK(grow_device(&a->str_pool, a->str_pool_n, cap));
        a->str_pool_cap = cap;
    }
    const unsigned long long base = a->list_n, pool_base = a->str_pool_n;
    a->list_n += (uint64_t)nrows;
    a->str_pool_n += nbytes;
    a->list_sorted = a->str_ready = false;
    if (nbytes)
        B200_CUDA(cudaMemcpyAsync(a->str_pool + pool_base, bytes, nbytes, cudaMemcpyDeviceToDevice, st));
    StrListParams p;
    memset(&p, 0, sizeof p);
    p.nb = nbinners;
    p.nrows = nrows;
    memcpy(p.b, db, sizeof(DevBinner) * nbinners);
    p.dropnull = (a->moment & 2) != 0; // AggList_string_int64(grid, grids, threads, dropnan, dropnull): dropnan (bit 0) has no effect
    p.offsets = offsets;
    p.first = first;
    p.nulls = nulls;
    p.keys = a->list_keys;
    p.vals = a->list_vals;
    p.start = a->str_start;
    p.base = base;
    p.pool_base = pool_base;
    p.skip_key = a->cells;
    const int blocks = nblocks_for(((unsigned long long)nrows + 3) / 4);
    if (vec)
        k_strlist_append<true><<<blocks, 256, 0, st>>>(p);
    else
        k_strlist_append<false><<<blocks, 256, 0, st>>>(p);
    B200_CUDA(cudaGetLastError());
    return B200_OK;
}

} // namespace b200

using namespace b200;

extern "C" {

/* sorts the records and reports the length of the flat value array (offsets[cells]); every slot is synchronised first */
int b200_agg_list_finish(b200_agg *a, int64_t *total_out) {
    if (!a || a->op != B200_AGG_LIST || !total_out) {
        set_error("b200_agg_list_finish: not a list aggregator");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CHECK(b200_ctx_sync(a->ctx, -1));
    std::lock_guard<std::mutex> g(a->nmu);
    cudaStream_t st = a->ctx->slots[0]->stream;
    const uint64_t n = a->list_n;
    if (!a->list_sorted && n > 1) {
        if (n >= (1ull << 32)) {
            set_error("AggList: more than 2^32 rows are not supported");
            return B200_ERR_UNSUPPORTED;
        }
        B200_CHECK(sort_records(a, st, a->cells * 4 + 3)); // keys are cell * 4 + category (skipped rows: cells * 4)
    }
    a->list_sorted = true;
    // per-cell counts -> offsets (kept on the device until read)
    const size_t cn = (size_t)a->cells + 1;
    if (!a->list_counts)
        B200_CUDA(cudaMalloc((void **)&a->list_counts, cn * 4));
    B200_CUDA(cudaMemsetAsync(a->list_counts, 0, cn * 4, st));
    if (n)
        k_list_count<<<nblocks_for(n), 256, 0, st>>>(a->list_keys, n, a->list_counts, a->cells);
    unsigned long long *d_total = nullptr;
    B200_CUDA(cudaMalloc((void **)&d_total, 8));
    k_scan_u32<<<1, 1024, 0, st>>>(a->list_counts, cn, d_total);
    B200_CUDA(cudaGetLastError());
    unsigned long long total = 0;
    B200_CUDA(cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    cudaFree(d_total);
    a->list_total = total;
    *total_out = (int64_t)total;
    return B200_OK;
}

/* after b200_agg_list_finish: offsets_out = int64[cells + 1], values_out = total elements of the aggregator's dtype */
int b200_agg_list_read(b200_agg *a, int64_t *offsets_out, void *values_out) {
    if (!a || a->op != B200_AGG_LIST || !offsets_out || !a->list_sorted || !a->list_counts) {
        set_error("b200_agg_list_read: call b200_agg_list_finish first");
        return B200_ERR_STATE;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    std::lock_guard<std::mutex> g(a->nmu);
    cudaStream_t st = a->ctx->slots[0]->stream;
    const size_t cn = (size_t)a->cells + 1;
    std::vector<unsigned> off(cn);
    B200_CUDA(cudaMemcpyAsync(off.data(), a->list_counts, cn * 4, cudaMemcpyDeviceToHost, st));
    const int isz = dtype_size(a->dtype);
    void *d_out = nullptr;
    if (a->list_total && values_out) {
        B200_CUDA(cudaMalloc(&d_out, a->list_total * isz));
        k_list_values<<<nblocks_for(a->list_total), 256, 0, st>>>(a->list_keys, a->list_vals, a->list_total, a->dtype, isz, d_out);
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaMemcpyAsync(values_out, d_out, a->list_total * isz, cudaMemcpyDeviceToHost, st));
    }
    B200_CUDA(cudaStreamSynchronize(st));
    cudaFree(d_out);
    for (size_t i = 0; i < cn; i++)
        offsets_out[i] = (int64_t)off[i];
    return B200_OK;
}

/* AggList_string: sorts the records (once), then builds the flat result on the device — list offsets, int64 string offsets, the
 * gathered bytes and the null flags — and reports its element and byte counts.  Calling it again without new rows skips the sort. */
int b200_agg_list_string_finish(b200_agg *a, int64_t *nelem_out, int64_t *nbytes_out) {
    if (!a || a->op != B200_AGG_LIST_STRING || !nelem_out || !nbytes_out) {
        set_error("b200_agg_list_string_finish: not a string list aggregator");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CHECK(b200_ctx_sync(a->ctx, -1));
    std::lock_guard<std::mutex> g(a->nmu);
    cudaStream_t st = a->ctx->slots[0]->stream;
    const uint64_t n = a->list_n;
    if (n >= (1ull << 32)) {
        set_error("AggList_string: more than 2^32 rows are not supported");
        return B200_ERR_UNSUPPORTED;
    }
    if (!a->list_sorted && n > 1)
        B200_CHECK(sort_records(a, st, a->cells)); // keys are cells (dropped nulls: cells)
    a->list_sorted = true;
    a->list_total = a->str_nbytes = 0;
    a->str_ready = false;
    struct Tmp {
        unsigned long long *p = nullptr;
        ~Tmp() { cudaFree(p); }
    } d_total, tile;
    // per-cell counts -> list offsets
    const size_t cn = (size_t)a->cells + 1;
    if (!a->list_counts)
        B200_CUDA(cudaMalloc((void **)&a->list_counts, cn * 4));
    B200_CUDA(cudaMemsetAsync(a->list_counts, 0, cn * 4, st));
    if (n)
        k_strlist_count<<<nblocks_for(n), 256, 0, st>>>(a->list_keys, n, a->list_counts, a->cells);
    B200_CUDA(cudaMalloc((void **)&d_total.p, 8));
    k_scan_u32<<<1, 1024, 0, st>>>(a->list_counts, cn, d_total.p);
    B200_CUDA(cudaGetLastError());
    unsigned long long total = 0, pool_end = a->str_pool_n;
    if (n) // the end of the last record's bytes
        B200_CUDA(cudaMemcpyAsync(a->str_start + n, &pool_end, 8, cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(&total, d_total.p, 8, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    // string offsets + null flags of the `total` leading (real) sorted records; the result buffers are kept and only ever grow
    // (a finish after a reset, or a second one, reuses them)
    if (total + 1 > a->str_elem_cap) {
        cudaFree(a->str_off);
        cudaFree(a->str_nulls);
        a->str_off = nullptr, a->str_nulls = nullptr, a->str_elem_cap = 0;
        B200_CUDA(cudaMalloc((void **)&a->str_off, (total + 1) * 8));
        B200_CUDA(cudaMalloc((void **)&a->str_nulls, total + 1));
        a->str_elem_cap = total + 1;
    }
    unsigned long long nbytes = 0;
    if (total) {
        const unsigned long long ntiles = (total + kStrTile - 1) / kStrTile;
        B200_CUDA(cudaMalloc((void **)&tile.p, ntiles * 8));
        k_strlist_tile_sums<<<(unsigned)ntiles, 256, 0, st>>>(a->list_vals, a->str_start, total, tile.p);
        k_scan_u64<<<1, 1024, 0, st>>>(tile.p, ntiles, reinterpret_cast<unsigned long long *>(a->str_off + total));
        k_strlist_offsets<<<(unsigned)ntiles, 256, 0, st>>>(a->list_vals, a->str_start, total, tile.p, a->str_off, a->str_nulls);
        B200_CUDA(cudaGetLastError());
        B200_CUDA(cudaMemcpyAsync(&nbytes, a->str_off + total, 8, cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
    } else {
        B200_CUDA(cudaMemsetAsync(a->str_off, 0, 8, st));
    }
    // the byte gather
    if (nbytes + 1 > a->str_bytes_cap) {
        cudaFree(a->str_bytes);
        a->str_bytes = nullptr, a->str_bytes_cap = 0;
        B200_CUDA(cudaMalloc((void **)&a->str_bytes, nbytes + 1));
        a->str_bytes_cap = nbytes + 1;
    }
    if (nbytes) {
        const unsigned long long warps = (total + 31) / 32;
        const int blocks = (int)std::max<unsigned long long>(1, std::min<unsigned long long>((warps + 7) / 8, 148ull * 16));
        k_strlist_gather<<<blocks, 256, 0, st>>>(a->list_vals, a->str_start, a->str_off, a->str_pool, total, a->str_bytes);
        B200_CUDA(cudaGetLastError());
    }
    B200_CUDA(cudaStreamSynchronize(st));
    a->list_total = total;
    a->str_nbytes = nbytes;
    a->str_ready = true;
    *nelem_out = (int64_t)total;
    *nbytes_out = (int64_t)nbytes;
    return B200_OK;
}

/* after b200_agg_list_string_finish, one D2H copy per buffer (any output may be NULL): list_offsets = int64[cells + 1],
 * str_offsets = int64[nelem + 1], bytes = nbytes, nulls = nelem flags (1 = null element) */
int b200_agg_list_string_read(b200_agg *a, int64_t *list_offsets, int64_t *str_offsets, uint8_t *bytes, uint8_t *nulls) {
    if (!a || a->op != B200_AGG_LIST_STRING || !a->list_sorted || !a->str_ready) {
        set_error("b200_agg_list_string_read: call b200_agg_list_string_finish first");
        return B200_ERR_STATE;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    std::lock_guard<std::mutex> g(a->nmu);
    cudaStream_t st = a->ctx->slots[0]->stream;
    const size_t cn = (size_t)a->cells + 1;
    std::vector<unsigned> off(list_offsets ? cn : 0);
    if (list_offsets)
        B200_CUDA(cudaMemcpyAsync(off.data(), a->list_counts, cn * 4, cudaMemcpyDeviceToHost, st));
    if (str_offsets)
        B200_CUDA(cudaMemcpyAsync(str_offsets, a->str_off, (a->list_total + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (bytes && a->str_nbytes)
        B200_CUDA(cudaMemcpyAsync(bytes, a->str_bytes, a->str_nbytes, cudaMemcpyDeviceToHost, st));
    if (nulls && a->list_total)
        B200_CUDA(cudaMemcpyAsync(nulls, a->str_nulls, a->list_total, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < off.size(); i++)
        list_offsets[i] = (int64_t)off[i];
    return B200_OK;
}

} // extern "C"
