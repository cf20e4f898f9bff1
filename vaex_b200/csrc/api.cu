// api.cu — the C ABI of libb200agg.so (include/b200agg.h): context/slots, aggregator objects, b200_bin.
#include <math.h>
#include <stdarg.h>

#include <immintrin.h>

#include <algorithm>
#include <chrono>

#include "binby.cuh"
#include "device_utils.cuh"

namespace b200 {

int set_fill_binner(b200_set *s, DevBinner &b); // hashset.cu

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    set_error("CUDA error %s (%s) at %s:%d in `%s`", cudaGetErrorName(e), cudaGetErrorString(e), file, line, what);
    return B200_ERR_CUDA;
}

// ---- staging of host chunks -----------------------------------------------------------------------
// Host column -> page-locked ring piece.  The piece is read next by the copy engine, not by a core: non-temporal stores keep it out
// of the caches and save the read-for-ownership of every destination line, which is what bounds glibc's memcpy when 16 feeder
// threads copy at once (measured: tools/probe_e2e_threads.py, profiles/r02_e2e_probe.txt).  `dst` is 64-byte aligned (the ring is
// page-locked memory, pieces start at multiples of the piece size); the sfence makes the stores visible before the DMA is enqueued.
__attribute__((target("avx2"))) static void copy_stream_avx2(char *dst, const char *src, size_t n) {
    size_t i = 0;
    for (; i + 128 <= n; i += 128) {
        const __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i));
        const __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i + 32));
        const __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i + 64));
        const __m256i d = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(src + i + 96));
        _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i), a);
        _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 32), b);
        _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 64), c);
        _mm256_stream_si256(reinterpret_cast<__m256i *>(dst + i + 96), d);
    }
    _mm_sfence();
    if (i < n)
        memcpy(dst + i, src + i, n - i);
}

static void copy_to_ring(void *dst, const void *src, size_t n) {
    static const bool avx2 = __builtin_cpu_supports("avx2") && !(getenv("B200_BOUNCE_MEMCPY") && atoi(getenv("B200_BOUNCE_MEMCPY")));
    if (avx2 && (reinterpret_cast<uintptr_t>(dst) & 31) == 0)
        copy_stream_avx2(static_cast<char *>(dst), static_cast<const char *>(src), n);
    else
        memcpy(dst, src, n);
}

int slot_reserve(b200_ctx *ctx, Slot *s, size_t bytes) {
    if (bytes <= s->stage_cap)
        return B200_OK;
    if (s->stage) {
        B200_CUDA(cudaStreamSynchronize(s->stream));
        B200_CUDA(cudaFree(s->stage));
        s->stage = nullptr;
        s->stage_cap = 0;
    }
    size_t cap = align_up(bytes + bytes / 4, 1 << 20);
    B200_CUDA(cudaMalloc(&s->stage, cap));
    s->stage_cap = cap;
    (void)ctx;
    return B200_OK;
}

// size classes of the cache: exact (256-byte granules) up to 1 MB, above that 8 steps per power of two (<= 12.5 % slack), so
// buffers whose size depends on a key count (hash tables, sort scratch) find a block again when the count moves a little
static size_t cache_class(size_t bytes) {
    bytes = align_up(bytes ? bytes : 1, 256);
    if (bytes <= (1u << 20))
        return bytes;
    size_t step = 1;
    while ((step << 4) <= bytes)
        step <<= 1; // step = 2^(floor(log2 bytes) - 3)
    return align_up(bytes, step);
}

cudaError_t ctx_alloc(b200_ctx *ctx, void **out, size_t bytes) {
    bytes = cache_class(bytes);
    {
        std::lock_guard<std::mutex> g(ctx->cache_mu);
        auto it = ctx->cache.find(bytes);
        if (it != ctx->cache.end()) {
            *out = it->second;
            ctx->cache.erase(it);
            ctx->cache_bytes -= bytes;
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e == cudaErrorMemoryAllocation) { // give the cache back before reporting out-of-memory
        cudaGetLastError();
        std::lock_guard<std::mutex> g(ctx->cache_mu);
        for (auto &kv : ctx->cache)
            cudaFree(kv.second);
        ctx->cache.clear();
        ctx->cache_bytes = 0;
        e = cudaMalloc(out, bytes);
    }
    return e;
}

void ctx_release(b200_ctx *ctx, void *p, size_t bytes) {
    if (!p)
        return;
    bytes = cache_class(bytes);
    constexpr size_t kCacheLimit = 4ull << 30; // per context; a block larger than a quarter of it is never kept
    {
        std::lock_guard<std::mutex> g(ctx->cache_mu);
        if (bytes <= kCacheLimit / 4 && ctx->cache_bytes + bytes <= kCacheLimit) {
            ctx->cache.emplace(bytes, p);
            ctx->cache_bytes += bytes;
            return;
        }
    }
    cudaFree(p);
}

bool is_device_pointer(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

void Stager::plan(const void *p, size_t bytes) {
    if (!p || memspace == B200_MEM_DEVICE)
        return;
    if (memspace == B200_MEM_MIXED && is_device_pointer(p))
        return;
    for (auto &e : entries)
        if (e.host == p) { // the same column used twice (e.g. binby x and sum x) is copied once
            e.bytes = std::max(e.bytes, bytes);
            return;
        }
    entries.push_back(Entry{p, bytes, nullptr});
}

int Stager::commit() {
    if (memspace == B200_MEM_DEVICE || entries.empty())
        return B200_OK;
    need = 0;
    for (auto &e : entries)
        need += align_up(e.bytes, 256);
    B200_CHECK(slot_reserve(ctx, slot, need));
    size_t off = 0;
    // MIXED keeps per-column copies (some columns are device pointers and were not planned); HOST chunks whose buffers die with
    // the call go through the slot's page-locked bounce ring
    const bool bounce = !async_host && memspace == B200_MEM_HOST;
    if (bounce) {
        // B200_BOUNCE_PIECE_KB / B200_BOUNCE_COUNT: ring geometry (defaults 4 MB x 4)
        static const size_t piece = getenv("B200_BOUNCE_PIECE_KB") ? std::max<size_t>(64, atol(getenv("B200_BOUNCE_PIECE_KB"))) << 10 : 4u << 20;
        static const unsigned count = getenv("B200_BOUNCE_COUNT") ? std::min<unsigned>(Slot::kBounceMax, std::max(2, atoi(getenv("B200_BOUNCE_COUNT")))) : 4u;
        using clk = std::chrono::steady_clock;
        auto ns = [](clk::time_point a, clk::time_point b) { return (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(b - a).count(); };
        for (auto &e : entries) {
            e.dev = static_cast<char *>(slot->stage) + off;
            for (size_t q = 0; q < e.bytes; q += piece) {
                const size_t len = std::min(piece, e.bytes - q);
                const unsigned b = slot->bounce_next++ % count;
                const auto t0 = clk::now();
                if (slot->bounce_cap[b] < piece) {
                    if (slot->bounce[b]) {
                        B200_CUDA(cudaEventSynchronize(slot->bounce_done[b]));
                        B200_CUDA(cudaFreeHost(slot->bounce[b]));
                        slot->bounce[b] = nullptr, slot->bounce_cap[b] = 0;
                    }
                    B200_CUDA(cudaHostAlloc(&slot->bounce[b], piece, cudaHostAllocPortable));
                    slot->bounce_cap[b] = piece;
                    if (!slot->bounce_done[b])
                        B200_CUDA(cudaEventCreateWithFlags(&slot->bounce_done[b], cudaEventDisableTiming));
                } else {
                    B200_CUDA(cudaEventSynchronize(slot->bounce_done[b])); // the copy that last read this piece has finished
                }
                const auto t1 = clk::now();
                copy_to_ring(slot->bounce[b], static_cast<const char *>(e.host) + q, len);
                const auto t2 = clk::now();
                B200_CUDA(cudaMemcpyAsync(static_cast<char *>(e.dev) + q, slot->bounce[b], len, cudaMemcpyHostToDevice, slot->stream));
                B200_CUDA(cudaEventRecord(slot->bounce_done[b], slot->stream));
                const auto t3 = clk::now();
                slot->host_ns[0] += ns(t0, t1), slot->host_ns[1] += ns(t1, t2), slot->host_ns[2] += ns(t2, t3), slot->host_pieces++;
            }
            off += align_up(e.bytes, 256);
        }
        return B200_OK;
    }
    for (auto &e : entries) {
        e.dev = static_cast<char *>(slot->stage) + off;
        off += align_up(e.bytes, 256);
        if (e.bytes)
            B200_CUDA(cudaMemcpyAsync(e.dev, e.host, e.bytes, cudaMemcpyHostToDevice, slot->stream));
    }
    return B200_OK;
}

const void *Stager::dev(const void *p) const {
    if (!p || memspace == B200_MEM_DEVICE)
        return p;
    for (auto &e : entries)
        if (e.host == p)
            return e.dev;
    return memspace == B200_MEM_MIXED ? p : nullptr; // MIXED: not planned == already on the device
}

// identity element of an aggregator's device cell
static uint64_t agg_init_bits(int op, int cell_dtype) {
    if (op != B200_AGG_MIN && op != B200_AGG_MAX)
        return 0;
    const bool mx = op == B200_AGG_MAX;
    switch (cell_dtype) {
    case B200_F64: return mx ? 0xfff0000000000000ULL : 0x7ff0000000000000ULL;
    case B200_F32: return mx ? 0xff800000u : 0x7f800000u;
    case B200_I64: return mx ? 0x8000000000000000ULL : 0x7fffffffffffffffULL;
    case B200_U64: return mx ? 0 : ~0ULL;
    case B200_I32: return mx ? 0x80000000u : 0x7fffffffu;
    default: return mx ? 0 : 0xffffffffu;
    }
}

// reference initial_fill for narrow min/max grids is numeric_limits<T>::min()/max() (src/agg_minmax.cpp:13-18,83-87);
// the device holds them widened to 32 bit, so untouched cells must come back as the narrow limit.
static int64_t narrow_limit(int dtype, bool mx) {
    switch (dtype) {
    case B200_I16: return mx ? INT16_MIN : INT16_MAX;
    case B200_I8: return mx ? INT8_MIN : INT8_MAX;
    case B200_U16: return mx ? 0 : UINT16_MAX;
    case B200_U8: return mx ? 0 : UINT8_MAX;
    case B200_BOOL: return mx ? 0 : 1;
    default: return 0;
    }
}

static int agg_fill(b200_agg *a, cudaStream_t st) {
    if (a->op == B200_AGG_LIST || a->op == B200_AGG_LIST_STRING) { // initial_fill: empty lists
        std::lock_guard<std::mutex> g(a->nmu);
        a->list_n = a->list_total = 0;
        a->str_pool_n = 0;
        a->str_ready = false;
        a->list_sorted = false;
        return B200_OK;
    }
    if (a->op == B200_AGG_NUNIQUE) {
        B200_CUDA(cudaMemsetAsync(a->grid, 0, (a->cells ? a->cells : 1) * 8 * 3, st));
        if (a->ntable)
            B200_CUDA(cudaMemsetAsync(a->ntable, 0xff, a->ncap * 16, st));
        B200_CUDA(cudaMemsetAsync(a->ntotal, 0, 8, st));
        a->npairs = 0;
        return B200_OK;
    }
    if (a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST) {
        // src/agg_first.cpp:19-26: value 99, order limits, cell_masked 1; the packed {key,row} state starts at the maximum
        const int isz = dtype_size(a->dtype), isz2 = dtype_size(a->dtype2);
        const bool inv = a->op == B200_AGG_LAST;
        auto bits_of = [](auto x) {
            uint64_t b = 0;
            memcpy(&b, &x, sizeof x);
            return b;
        };
        uint64_t vbits = 99, obits = 0;
        switch (a->dtype) {
        case B200_F64: vbits = bits_of(99.0); break;
        case B200_F32: vbits = bits_of(99.0f); break;
        case B200_BOOL: vbits = 1; break;
        default: break;
        }
        switch (a->dtype2) {
        case B200_F64: obits = bits_of(inv ? 2.2250738585072014e-308 : 1.7976931348623157e308); break;
        case B200_F32: obits = bits_of(inv ? 1.17549435e-38f : 3.40282347e38f); break;
        case B200_I64: obits = (uint64_t)(inv ? INT64_MIN : INT64_MAX); break;
        case B200_I32: obits = (uint32_t)(inv ? INT32_MIN : INT32_MAX); break;
        case B200_I16: obits = (uint16_t)(inv ? INT16_MIN : INT16_MAX); break;
        case B200_I8: obits = (uint8_t)(inv ? INT8_MIN : INT8_MAX); break;
        case B200_U64: obits = inv ? 0 : UINT64_MAX; break;
        case B200_U32: obits = inv ? 0 : UINT32_MAX; break;
        case B200_U16: obits = inv ? 0 : UINT16_MAX; break;
        case B200_U8: obits = inv ? 0 : UINT8_MAX; break;
        default: obits = inv ? 0 : 1; break;
        }
        // filled on the device, stream-ordered: no O(cells) host vectors, no host sync
        B200_CHECK(launch_fill_elems(st, a->grid, isz, a->cells, vbits));
        B200_CHECK(launch_fill_elems(st, a->order, isz2, a->cells, obits));
        B200_CUDA(cudaMemsetAsync(a->cell_masked, 1, a->cells, st));
        B200_CUDA(cudaMemsetAsync(a->state, 0xff, a->cells * 16, st));
        return B200_OK;
    }
    const uint64_t bits = agg_init_bits(a->op, a->cell_dtype);
    if (bits == 0)
        B200_CUDA(cudaMemsetAsync(a->grid, 0, a->cells * dtype_size(a->cell_dtype), st));
    else
        B200_CHECK(launch_fill(st, a->grid, a->cell_dtype, a->cells, bits));
    return B200_OK;
}

} // namespace b200

namespace b200 {
int bin_list(b200_ctx *ctx, Slot *sl, b200_agg *a, const DevBinner *db, int nbinners, const void *data, const uint8_t *mask, int64_t nrows, bool vec); // list.cu
int bin_list_string(Slot *sl, b200_agg *a, const DevBinner *db, int nbinners, const long long *offsets, const unsigned char *bytes, long long first,
                    unsigned long long nbytes, const uint8_t *nulls, int64_t nrows, bool vec); // list.cu
}

using namespace b200;

extern "C" {

const char *b200_last_error(void) { return g_err; }
int b200_abi_version(void) { return B200_ABI_VERSION; }

int b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int b200_ctx_create(int device, int nslots, b200_ctx **out) {
    if (!out || nslots < 1 || nslots > 1024) {
        set_error("b200_ctx_create: invalid argument");
        return B200_ERR_INVALID;
    }
    int ndev = 0;
    B200_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) {
        set_error("b200_ctx_create: device %d not present (%d CUDA devices) — this library has no CPU fallback", device, ndev);
        return B200_ERR_CUDA;
    }
    B200_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    B200_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("b200_ctx_create: device %d is sm_%d%d; libb200agg is built for sm_100a only", device, prop.major, prop.minor);
        return B200_ERR_CUDA;
    }
    b200_ctx *ctx = new b200_ctx;
    ctx->device = device;
    ctx->nslots = nslots;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    for (int i = 0; i < nslots; i++) {
        Slot *s = new Slot;
        ctx->slots.push_back(s); // owned by ctx from here on: a failure below is undone by b200_ctx_destroy
        cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
        if (e == cudaSuccess)
            e = cudaEventCreateWithFlags(&s->h2d_done, cudaEventDisableTiming);
        if (e == cudaSuccess)
            e = cudaMallocHost(&s->pinned, 4096);
        if (e == cudaSuccess)
            e = cudaMalloc(&s->dscratch, 4096);
        if (e != cudaSuccess) {
            b200_ctx_destroy(ctx);
            return cuda_fail(e, "b200_ctx_create: slot resources", __FILE__, __LINE__);
        }
    }
    *out = ctx;
    return B200_OK;
}

int b200_ctx_destroy(b200_ctx *ctx) {
    if (!ctx)
        return B200_OK;
    cudaSetDevice(ctx->device);
    for (Slot *s : ctx->slots) {
        if (s->stream)
            cudaStreamSynchronize(s->stream);
        cudaFree(s->stage);
        cudaFree(s->scratch);
        cudaFree(s->dscratch);
        cudaFreeHost(s->pinned);
        for (int b = 0; b < Slot::kBounceMax; b++) {
            if (s->bounce[b])
                cudaFreeHost(s->bounce[b]);
            if (s->bounce_done[b])
                cudaEventDestroy(s->bounce_done[b]);
        }
        if (s->h2d_done)
            cudaEventDestroy(s->h2d_done);
        if (s->stream)
            cudaStreamDestroy(s->stream);
        delete s;
    }
    for (auto &kv : ctx->cache)
        cudaFree(kv.second);
    delete ctx;
    return B200_OK;
}

int b200_ctx_sync(b200_ctx *ctx, int slot) {
    if (!ctx || slot >= ctx->nslots) {
        set_error("b200_ctx_sync: invalid argument");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(ctx->device));
    if (slot < 0) {
        for (Slot *s : ctx->slots)
            B200_CUDA(cudaStreamSynchronize(s->stream));
    } else {
        B200_CUDA(cudaStreamSynchronize(ctx->slots[slot]->stream));
    }
    return B200_OK;
}

int b200_ctx_device(const b200_ctx *ctx) { return ctx ? ctx->device : -1; }

int b200_host_register(const void *ptr, size_t bytes) {
    if (!ptr || !bytes) {
        set_error("b200_host_register: invalid argument");
        return B200_ERR_INVALID;
    }
    cudaError_t e = cudaHostRegister(const_cast<void *>(ptr), bytes, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) {
        cudaGetLastError();
        return B200_OK;
    }
    B200_CUDA(e);
    return B200_OK;
}

int b200_host_unregister(const void *ptr) {
    cudaError_t e = cudaHostUnregister(const_cast<void *>(ptr));
    if (e == cudaErrorHostMemoryNotRegistered) {
        cudaGetLastError();
        return B200_OK;
    }
    B200_CUDA(e);
    return B200_OK;
}

int b200_ctx_stream(b200_ctx *ctx, int slot, void **stream_out) {
    if (!ctx || slot < 0 || slot >= ctx->nslots || !stream_out) {
        set_error("b200_ctx_stream: invalid argument");
        return B200_ERR_INVALID;
    }
    *stream_out = (void *)ctx->slots[slot]->stream;
    return B200_OK;
}

int b200_ctx_path_stats(b200_ctx *ctx, int slot, uint64_t out[6]) {
    if (!ctx || slot < 0 || slot >= ctx->nslots || !out) {
        set_error("b200_ctx_path_stats: invalid argument");
        return B200_ERR_INVALID;
    }
    Slot *s = ctx->slots[slot];
    memset(out, 0, 6 * sizeof(uint64_t));
    B200_CUDA(cudaSetDevice(ctx->device));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    const char *lo = static_cast<const char *>(s->scratch), *hi = lo + s->scratch_cap;
    const char *q = reinterpret_cast<const char *>(s->ring_len);
    if (!q || q < lo || q + s->ring_lists * 4 > hi) // never ran, or the scratch was reallocated since
        return B200_OK;
    std::vector<unsigned> len(s->ring_lists);
    unsigned chunks = 0;
    B200_CUDA(cudaMemcpy(len.data(), s->ring_len, s->ring_lists * 4, cudaMemcpyDeviceToHost));
    B200_CUDA(cudaMemcpy(&chunks, s->ring_ctl, 4, cudaMemcpyDeviceToHost));
    uint64_t entries = 0;
    for (unsigned v : len)
        entries += v;
    out[0] = s->ring_rows, out[1] = entries, out[2] = chunks, out[3] = s->ring_chunk_entries, out[4] = s->ring_memset_bytes, out[5] = s->ring_lists;
    return B200_OK;
}

namespace {
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__global__ void k_spin(unsigned long long ns) {
    extern __shared__ unsigned char spin_smem[];
    const unsigned long long t0 = globaltimer_ns();
    while (globaltimer_ns() - t0 < ns)
        __nanosleep(200);
    if (ns == ~0ull)
        spin_smem[threadIdx.x] = 0;
}
} // namespace

int b200_ctx_occupy(b200_ctx *ctx, int slot, int ctas, int threads, int smem_bytes, uint64_t nanoseconds) {
    if (!ctx || slot < 0 || slot >= ctx->nslots || ctas < 1 || threads < 1 || threads > 1024 || smem_bytes < 0) {
        set_error("b200_ctx_occupy: invalid argument");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(ctx->device));
    B200_CUDA(cudaFuncSetAttribute(k_spin, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    k_spin<<<ctas, threads, smem_bytes, ctx->slots[slot]->stream>>>(nanoseconds);
    B200_CUDA(cudaGetLastError());
    return B200_OK;
}

int b200_ctx_host_stats(b200_ctx *ctx, uint64_t out[6], int reset) {
    if (!ctx || !out) {
        set_error("b200_ctx_host_stats: invalid argument");
        return B200_ERR_INVALID;
    }
    memset(out, 0, 6 * sizeof(uint64_t));
    for (Slot *s : ctx->slots) {
        std::lock_guard<std::mutex> g(s->mu);
        for (int k = 0; k < 4; k++)
            out[k] += s->host_ns[k];
        out[4] += s->host_pieces, out[5] += s->host_calls;
        if (reset)
            s->host_ns[0] = s->host_ns[1] = s->host_ns[2] = s->host_ns[3] = s->host_pieces = s->host_calls = 0;
    }
    return B200_OK;
}

// ---- aggregators -----------------------------------------------------------------------------------
static bool is_list(int op) { return op == B200_AGG_LIST || op == B200_AGG_LIST_STRING; }
static size_t agg_cells_alloc(const b200_agg *a) { return is_list(a->op) ? 16 : (a->cells ? a->cells : 1); }
static size_t agg_grid_bytes(const b200_agg *a) { return agg_cells_alloc(a) * dtype_size(a->cell_dtype) * (a->op == B200_AGG_NUNIQUE ? 3 : 1); }

int b200_agg_create(b200_ctx *ctx, int op, int dtype, int dtype2, int byteswap, uint32_t moment, uint64_t cells, b200_agg **out) {
    if (!ctx || !out || op < B200_AGG_COUNT || op > B200_AGG_LIST_STRING || dtype < 0 || dtype >= B200_NDTYPE || dtype2 < 0 || dtype2 >= B200_NDTYPE) {
        set_error("b200_agg_create: invalid argument");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(ctx->device));
    b200_agg *a = new b200_agg;
    a->ctx = ctx;
    a->op = op;
    a->dtype = dtype;
    a->dtype2 = dtype2;
    a->byteswap = byteswap;
    a->moment = moment;
    a->cells = cells;
    switch (op) {
    case B200_AGG_COUNT:
    case B200_AGG_NUNIQUE: a->cell_dtype = B200_I64; break;
    case B200_AGG_LIST:
    case B200_AGG_LIST_STRING: a->cell_dtype = B200_U8; break; // no cell-shaped state: records are appended (list.cu)
    case B200_AGG_SUM:
    case B200_AGG_SUM_MOMENT: a->cell_dtype = dtype_upcast(dtype); break;
    case B200_AGG_MIN:
    case B200_AGG_MAX: a->cell_dtype = dtype_minmax_cell(dtype); break;
    default: a->cell_dtype = dtype; break;
    }
    const size_t n = is_list(op) ? 16 : (cells ? cells : 1);
    cudaError_t e = ctx_alloc(ctx, &a->grid, agg_grid_bytes(a));
    if (e == cudaSuccess && op == B200_AGG_NUNIQUE)
        e = cudaMalloc((void **)&a->ntotal, 8);
    if (e == cudaSuccess && (op == B200_AGG_FIRST || op == B200_AGG_LAST)) {
        e = ctx_alloc(ctx, &a->state, n * 16);
        if (e == cudaSuccess)
            e = ctx_alloc(ctx, &a->order, n * dtype_size(dtype2));
        if (e == cudaSuccess)
            e = ctx_alloc(ctx, (void **)&a->cell_masked, n);
        if (e == cudaSuccess)
            e = cudaEventCreateWithFlags(&a->chain, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        b200_agg_destroy(a);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            set_error("b200_agg_create: out of device memory for %llu cells", (unsigned long long)cells);
            return B200_ERR_NOMEM;
        }
        return cuda_fail(e, "cudaMalloc(grid)", __FILE__, __LINE__);
    }
    cudaStream_t st = ctx->slots[0]->stream;
    int rc = agg_fill(a, st);
    if (!rc && cudaStreamSynchronize(st) != cudaSuccess)
        rc = B200_ERR_CUDA;
    if (rc) {
        b200_agg_destroy(a);
        return rc;
    }
    *out = a;
    return B200_OK;
}

int b200_agg_destroy(b200_agg *a) {
    if (!a)
        return B200_OK;
    cudaSetDevice(a->ctx->device);
    // the cell-shaped buffers go back to the context's cache: nothing in flight may still touch them
    for (Slot *s : a->ctx->slots)
        cudaStreamSynchronize(s->stream);
    const size_t n = agg_cells_alloc(a);
    ctx_release(a->ctx, a->grid, agg_grid_bytes(a));
    ctx_release(a->ctx, a->state, n * 16);
    ctx_release(a->ctx, a->order, n * dtype_size(a->dtype2));
    ctx_release(a->ctx, a->cell_masked, n);
    cudaFree(a->ntable);
    cudaFree(a->ntotal);
    cudaFree(a->list_keys);
    cudaFree(a->list_vals);
    cudaFree(a->list_counts);
    cudaFree(a->str_pool);
    cudaFree(a->str_start);
    cudaFree(a->str_off);
    cudaFree(a->str_bytes);
    cudaFree(a->str_nulls);
    if (a->chain)
        cudaEventDestroy(a->chain);
    delete a;
    return B200_OK;
}

int b200_agg_reset(b200_agg *a) {
    if (!a) {
        set_error("b200_agg_reset: null");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CHECK(b200_ctx_sync(a->ctx, -1));
    cudaStream_t st = a->ctx->slots[0]->stream;
    B200_CHECK(agg_fill(a, st));
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_agg_reset_on(b200_agg *a, int slot) {
    if (!a || slot < 0 || slot >= a->ctx->nslots) {
        set_error("b200_agg_reset_on: invalid argument");
        return B200_ERR_INVALID;
    }
    if (a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST || a->op == B200_AGG_NUNIQUE)
        return b200_agg_reset(a);
    B200_CUDA(cudaSetDevice(a->ctx->device));
    return agg_fill(a, a->ctx->slots[slot]->stream);
}

int b200_agg_read_on(b200_agg *a, int slot, void *values_out) {
    if (!a || !values_out || slot < 0 || slot >= a->ctx->nslots) {
        set_error("b200_agg_read_on: invalid argument");
        return B200_ERR_INVALID;
    }
    if (a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST || a->op == B200_AGG_NUNIQUE || is_list(a->op)) {
        set_error("b200_agg_read_on: not available for first/last/nunique/list");
        return B200_ERR_UNSUPPORTED;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CUDA(cudaMemcpyAsync(values_out, a->grid, a->cells * dtype_size(a->cell_dtype), cudaMemcpyDeviceToHost, a->ctx->slots[slot]->stream));
    return B200_OK;
}

uint64_t b200_agg_cells(const b200_agg *a) { return a ? a->cells : 0; }

int b200_agg_result_dtype(const b200_agg *a) {
    switch (a->op) {
    case B200_AGG_COUNT:
    case B200_AGG_NUNIQUE: return B200_I64;
    case B200_AGG_SUM:
    case B200_AGG_SUM_MOMENT: return dtype_upcast(a->dtype);
    default: return a->dtype;
    }
}

size_t b200_agg_bytes(const b200_agg *a) { return (size_t)dtype_size(b200_agg_result_dtype(a)) * a->cells; }
int b200_agg_device_dtype(const b200_agg *a) { return a->cell_dtype; }

int b200_agg_device_ptr(b200_agg *a, int which, void **ptr, size_t *bytes) {
    if (!a || !ptr || which < 0 || which > 3) {
        set_error("b200_agg_device_ptr: invalid argument");
        return B200_ERR_INVALID;
    }
    size_t n = 0;
    switch (which) {
    case 0:
        *ptr = a->grid;
        n = a->cells * dtype_size(a->cell_dtype) * (a->op == B200_AGG_NUNIQUE ? 3 : 1);
        break;
    case 1:
        *ptr = a->state;
        n = a->state ? a->cells * 16 : 0;
        break;
    case 2:
        *ptr = a->order;
        n = a->order ? a->cells * dtype_size(a->dtype2) : 0;
        break;
    default:
        *ptr = a->cell_masked;
        n = a->cell_masked ? a->cells : 0;
        break;
    }
    if (bytes)
        *bytes = n;
    return B200_OK;
}

int b200_agg_read(b200_agg *a, void *values_out, uint8_t *cell_masked_out) {
    if (!a || !values_out) {
        set_error("b200_agg_read: invalid argument");
        return B200_ERR_INVALID;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CHECK(b200_ctx_sync(a->ctx, -1));
    if (is_list(a->op)) {
        set_error("b200_agg_read: list aggregators are read with b200_agg_list[_string]_finish / b200_agg_list[_string]_read");
        return B200_ERR_UNSUPPORTED;
    }
    const int rdt = b200_agg_result_dtype(a);
    const int rsz = dtype_size(rdt), csz = dtype_size(a->cell_dtype);
    if (!a->cells)
        return B200_OK;
    if (a->op == B200_AGG_NUNIQUE) {
        // src/agg_nunique.cpp:16-42: counter.count() = keys + (any null) + (any NaN); dropmissing / dropnan subtract the NUMBER OF
        // null / NaN ROWS of the cell (null_count / nan_count are row counts there) — reproduced as is
        std::vector<uint64_t> planes(a->cells * 3);
        B200_CUDA(cudaMemcpy(planes.data(), a->grid, a->cells * 24, cudaMemcpyDeviceToHost));
        int64_t *out = static_cast<int64_t *>(values_out);
        for (uint64_t i = 0; i < a->cells; i++) {
            const int64_t nan = (int64_t)planes[a->cells + i], null = (int64_t)planes[2 * a->cells + i];
            int64_t c = (int64_t)planes[i] + (null > 0) + (nan > 0);
            if (a->moment & 1)
                c -= null;
            if (a->moment & 2)
                c -= nan;
            out[i] = c;
        }
        if (cell_masked_out)
            memset(cell_masked_out, 0, a->cells);
        return B200_OK;
    }
    if (rsz == csz) {
        B200_CUDA(cudaMemcpy(values_out, a->grid, a->cells * rsz, cudaMemcpyDeviceToHost));
    } else {
        // narrow min/max grids: 32-bit device cells -> 8/16-bit result; untouched cells map to the narrow limit
        std::vector<uint32_t> tmp(a->cells);
        B200_CUDA(cudaMemcpy(tmp.data(), a->grid, a->cells * 4, cudaMemcpyDeviceToHost));
        const bool mx = a->op == B200_AGG_MAX;
        const uint32_t init = (uint32_t)agg_init_bits(a->op, a->cell_dtype);
        const int64_t lim = narrow_limit(a->dtype, mx);
        for (uint64_t i = 0; i < a->cells; i++) {
            int64_t v = tmp[i] == init ? lim : (a->cell_dtype == B200_I32 ? (int64_t)(int32_t)tmp[i] : (int64_t)tmp[i]);
            if (rsz == 2)
                static_cast<uint16_t *>(values_out)[i] = (uint16_t)v;
            else
                static_cast<uint8_t *>(values_out)[i] = (uint8_t)v;
        }
    }
    if (cell_masked_out) {
        if (a->cell_masked)
            B200_CUDA(cudaMemcpy(cell_masked_out, a->cell_masked, a->cells, cudaMemcpyDeviceToHost));
        else
            memset(cell_masked_out, 0, a->cells);
    }
    return B200_OK;
}

int b200_agg_write(b200_agg *a, const void *values) {
    if (!a || !values) {
        set_error("b200_agg_write: invalid argument");
        return B200_ERR_INVALID;
    }
    if (a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST || a->op == B200_AGG_NUNIQUE || a->op == B200_AGG_LIST_STRING) {
        set_error("b200_agg_write: first/last/nunique/string list grids cannot be loaded (no per-cell state)");
        return B200_ERR_UNSUPPORTED;
    }
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CHECK(b200_ctx_sync(a->ctx, -1));
    const int rsz = dtype_size(b200_agg_result_dtype(a)), csz = dtype_size(a->cell_dtype);
    if (rsz == csz) {
        B200_CUDA(cudaMemcpy(a->grid, values, a->cells * rsz, cudaMemcpyHostToDevice));
    } else {
        std::vector<uint32_t> tmp(a->cells);
        for (uint64_t i = 0; i < a->cells; i++) {
            if (a->cell_dtype == B200_I32)
                tmp[i] = (uint32_t)(int32_t)(rsz == 2 ? (int32_t) static_cast<const int16_t *>(values)[i] : (int32_t) static_cast<const int8_t *>(values)[i]);
            else
                tmp[i] = rsz == 2 ? static_cast<const uint16_t *>(values)[i] : static_cast<const uint8_t *>(values)[i];
        }
        B200_CUDA(cudaMemcpy(a->grid, tmp.data(), a->cells * 4, cudaMemcpyHostToDevice));
    }
    return B200_OK;
}

namespace {
struct DeviceTemp {
    void *p = nullptr;
    ~DeviceTemp() { cudaFree(p); }
};
} // namespace

int b200_agg_merge(b200_agg *a, b200_agg *const *others, int nothers) {
    if (!a || (nothers && !others)) {
        set_error("b200_agg_merge: invalid argument");
        return B200_ERR_INVALID;
    }
    if (a->op == B200_AGG_NUNIQUE && nothers) {
        set_error("merge not implemented"); // src/agg_nunique.cpp:43-46
        return B200_ERR_UNSUPPORTED;
    }
    if (is_list(a->op))
        return B200_OK; // AggListPrimitive::merge / AggListString::merge are empty (src/agg_list.cpp:45, :140)
    B200_CUDA(cudaSetDevice(a->ctx->device));
    B200_CHECK(b200_ctx_sync(a->ctx, -1));
    cudaStream_t st = a->ctx->slots[0]->stream;
    for (int i = 0; i < nothers; i++) {
        b200_agg *o = others[i];
        if (o->op != a->op || o->dtype != a->dtype || o->cells != a->cells || o->dtype2 != a->dtype2) {
            set_error("b200_agg_merge: aggregators differ");
            return B200_ERR_INVALID;
        }
        if (o->ctx != a->ctx)
            B200_CHECK(b200_ctx_sync(o->ctx, -1));
        // same-process peers on other devices are read through UVA peer access when enabled; keep it simple: stage through host
        const void *src = o->grid;
        DeviceTemp tmp_, tstate_, torder_, tmask_; // freed on every way out of this iteration
        void *&tmp = tmp_.p, *&tstate = tstate_.p, *&torder = torder_.p, *&tmask = tmask_.p;
        b200_agg view; // shallow alias of `o` (b200_agg is not copyable: it owns a mutex)
        view.ctx = o->ctx, view.op = o->op, view.dtype = o->dtype, view.dtype2 = o->dtype2, view.byteswap = o->byteswap, view.moment = o->moment;
        view.cells = o->cells, view.cell_dtype = o->cell_dtype, view.grid = o->grid, view.state = o->state, view.order = o->order, view.cell_masked = o->cell_masked;
        if (o->ctx->device != a->ctx->device) {
            const size_t nb = o->cells * dtype_size(o->cell_dtype);
            B200_CUDA(cudaMalloc(&tmp, nb ? nb : 1));
            B200_CUDA(cudaMemcpyPeer(tmp, a->ctx->device, o->grid, o->ctx->device, nb));
            src = tmp;
            view.grid = tmp;
            if (o->state) {
                B200_CUDA(cudaMalloc(&tstate, o->cells * 16));
                B200_CUDA(cudaMemcpyPeer(tstate, a->ctx->device, o->state, o->ctx->device, o->cells * 16));
                B200_CUDA(cudaMalloc(&torder, o->cells * dtype_size(o->dtype2)));
                B200_CUDA(cudaMemcpyPeer(torder, a->ctx->device, o->order, o->ctx->device, o->cells * dtype_size(o->dtype2)));
                B200_CUDA(cudaMalloc(&tmask, o->cells));
                B200_CUDA(cudaMemcpyPeer(tmask, a->ctx->device, o->cell_masked, o->ctx->device, o->cells));
                view.state = tstate;
                view.order = torder;
                view.cell_masked = static_cast<uint8_t *>(tmask);
            }
        }
        int rc;
        if (a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST)
            rc = launch_merge_first(st, a, &view);
        else
            rc = launch_merge(st, a->op, a->cell_dtype, a->grid, src, a->cells);
        if (!rc && cudaStreamSynchronize(st) != cudaSuccess)
            rc = B200_ERR_CUDA;
        B200_CHECK(rc);
    }
    return B200_OK;
}

// ---- the hot path ----------------------------------------------------------------------------------
// NUNIQUE: batches of rows; before every launch the pair table is made large enough for (pairs so far + rows of the batch) at
// load <= 0.5, so an insert can never fail inside the kernel.  Callers on several slots share one table: serialised here.
static int bin_nunique(b200_ctx *ctx, Slot *sl, b200_agg *a, const DevBinner *db, int nbinners, const void *data, const uint8_t *valid,
                       const uint8_t *selection, int64_t nrows, bool vec) {
    std::lock_guard<std::mutex> g(a->nmu);
    cudaStream_t st = sl->stream;
    NUniqueParams np;
    memset(&np, 0, sizeof np);
    np.nb = nbinners;
    memcpy(np.b, db, sizeof(DevBinner) * nbinners);
    np.dtype = a->dtype;
    np.isz = dtype_size(a->dtype);
    np.byteswap = a->byteswap && np.isz > 1;
    np.data = data;
    np.valid = valid;
    np.selection = selection;
    np.distinct = static_cast<unsigned long long *>(a->grid);
    np.nan_rows = np.distinct + a->cells;
    np.null_rows = np.distinct + 2 * a->cells;
    np.total = a->ntotal;
    bool v = vec && !(reinterpret_cast<uintptr_t>(data) & 15) && !(reinterpret_cast<uintptr_t>(valid) & 15) && !(reinterpret_cast<uintptr_t>(selection) & 15);
    const int64_t batch = 1ll << 24;
    for (int64_t r0 = 0; r0 < nrows; r0 += batch) {
        const int64_t n = std::min<int64_t>(batch, nrows - r0);
        uint64_t need = 1 << 12;
        while (need < 2 * (a->npairs + (uint64_t)n))
            need <<= 1;
        if (need > a->ncap) {
            unsigned long long *nt = nullptr;
            cudaError_t e = cudaMalloc((void **)&nt, need * 16);
            if (e != cudaSuccess) {
                cudaGetLastError();
                set_error("nunique: out of device memory for a table of %llu slots", (unsigned long long)need);
                return B200_ERR_NOMEM;
            }
            B200_CUDA(cudaMemsetAsync(nt, 0xff, need * 16, st));
            if (a->ntable) {
                B200_CHECK(launch_nunique_rehash(st, a->ntable, a->ncap, nt, need));
                B200_CUDA(cudaStreamSynchronize(st));
                cudaFree(a->ntable);
            }
            a->ntable = nt;
            a->ncap = need;
        }
        np.table = a->ntable;
        np.tmask = a->ncap - 1;
        np.row0 = r0;
        np.nrows = n;
        B200_CHECK(launch_nunique(ctx, st, np, v));
        unsigned long long total = 0;
        B200_CUDA(cudaMemcpyAsync(&total, a->ntotal, 8, cudaMemcpyDeviceToHost, st));
        B200_CUDA(cudaStreamSynchronize(st));
        a->npairs = total;
    }
    return B200_OK;
}

int b200_bin(b200_ctx *ctx, int slot, const b200_binner *binners, int nbinners, const b200_agg_input *aggs, int naggs, int64_t nrows,
             int64_t row_offset, int memspace, uint32_t flags) {
    if (!ctx || slot < 0 || slot >= ctx->nslots || nbinners < 0 || nbinners > B200_MAX_BINNERS || naggs < 0 || nrows < 0 || (nbinners && !binners) ||
        (naggs && !aggs)) {
        set_error("b200_bin: invalid argument (slot %d of %d, %d binners, %d aggregators, %lld rows)", slot, ctx ? ctx->nslots : 0, nbinners, naggs,
                  (long long)nrows);
        return B200_ERR_INVALID;
    }
    if (nrows == 0 || naggs == 0)
        return B200_OK;
    B200_CUDA(cudaSetDevice(ctx->device));

    // grid layout: first binner fastest (src/agg.hpp:63-73)
    DevBinner db[B200_MAX_BINNERS];
    unsigned long long cells = 1;
    for (int i = 0; i < nbinners; i++) {
        const b200_binner &b = binners[i];
        DevBinner &d = db[i];
        memset(&d, 0, sizeof d);
        if (b.dtype < 0 || b.dtype >= B200_NDTYPE || !b.data) {
            set_error("b200_bin: binner %d: %s", i, b.data ? "unknown dtype" : "data not set");
            return b.data ? B200_ERR_INVALID : B200_ERR_NODATA;
        }
        d.kind = b.kind;
        d.dtype = b.dtype;
        d.isz = dtype_size(b.dtype);
        d.byteswap = b.byteswap && d.isz > 1;
        d.allow_other = b.allow_other;
        d.invert = b.invert;
        d.stride = cells;
        unsigned long long shape;
        if (b.kind == B200_BINNER_SCALAR) {
            d.vmin = b.vmin;
            d.scale = 1. / (b.vmax - b.vmin); // const double scale_v = 1. / (vmax - vmin)  (src/binners.cpp:16)
            d.bins = b.bins;
            d.bins_d = (double)b.bins;
            shape = b.bins + 3;
        } else if (b.kind == B200_BINNER_ORDINAL || b.kind == B200_BINNER_HASH) {
            d.ordinal_count = b.ordinal_count;
            d.min_value = b.min_value;
            shape = (unsigned long long)b.ordinal_count + (b.allow_other ? 3 : 2);
            if (b.kind == B200_BINNER_HASH) {
                if (!b.set) {
                    set_error("b200_bin: binner %d: hash binner without a set", i);
                    return B200_ERR_INVALID;
                }
                d.byteswap = 0;
                B200_CHECK(set_fill_binner(const_cast<b200_set *>(b.set), d));
            } else {
                d.byteswap = b.byteswap != 0; // the ordinal FlipEndian quirk flips the int64 difference, any itemsize
            }
        } else {
            set_error("b200_bin: binner %d: unknown kind %d", i, b.kind);
            return B200_ERR_INVALID;
        }
        cells *= shape;
    }
    for (int k = 0; k < naggs; k++) {
        if (!aggs[k].agg) {
            set_error("b200_bin: aggregator %d is null", k);
            return B200_ERR_INVALID;
        }
        if (aggs[k].agg->cells != cells) {
            set_error("b200_bin: aggregator %d has %llu cells, the binners span %llu", k, (unsigned long long)aggs[k].agg->cells, cells);
            return B200_ERR_INVALID;
        }
        if (!aggs[k].data && aggs[k].agg->op != B200_AGG_COUNT) {
            set_error("data not set"); // src/agg_sum.cpp:101-103, src/agg_minmax.cpp:50-52
            return B200_ERR_NODATA;
        }
    }

    Slot *sl = ctx->slots[slot];
    std::lock_guard<std::mutex> guard(sl->mu);
    cudaStream_t st = sl->stream;
    struct HostTimer { // wall time of HOST calls on this slot, for b200_ctx_host_stats
        Slot *s;
        std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
        ~HostTimer() {
            if (s)
                s->host_ns[3] += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count(), s->host_calls++;
        }
    } host_timer{memspace == B200_MEM_HOST ? sl : nullptr};

    // stage host columns (each distinct pointer once)
    Stager stg{ctx, sl, memspace};
    stg.async_host = (flags & B200_FLAG_ASYNC_HOST) != 0;
    for (int i = 0; i < nbinners; i++) {
        stg.plan(binners[i].data, (size_t)nrows * db[i].isz);
        if (binners[i].mask)
            stg.plan(binners[i].mask, (size_t)nrows);
    }
    // string list aggregators (`data` = int64 offsets[nrows + 1], `order` = bytes): the call's bytes are offsets[0] .. offsets[nrows]
    // (a sliced arrow array starts past 0); only that range is staged, indexed with offsets[j] - offsets[0]
    std::vector<long long> str_first(naggs, 0), str_nbytes(naggs, 0);
    for (int k = 0; k < naggs; k++) {
        const b200_agg *a = aggs[k].agg;
        if (a->op == B200_AGG_LIST_STRING) {
            const long long *off = static_cast<const long long *>(aggs[k].data);
            long long ends[2] = {0, 0};
            if (memspace == B200_MEM_DEVICE || (memspace == B200_MEM_MIXED && is_device_pointer(off))) {
                B200_CUDA(cudaMemcpyAsync(&ends[0], off, 8, cudaMemcpyDeviceToHost, st));
                B200_CUDA(cudaMemcpyAsync(&ends[1], off + nrows, 8, cudaMemcpyDeviceToHost, st));
                B200_CUDA(cudaStreamSynchronize(st));
            } else {
                ends[0] = off[0], ends[1] = off[nrows];
            }
            if (ends[1] < ends[0] || (ends[1] > ends[0] && !aggs[k].order)) {
                set_error("b200_bin: string list aggregator %d: invalid string offsets or bytes not set", k);
                return B200_ERR_INVALID;
            }
            str_first[k] = ends[0], str_nbytes[k] = ends[1] - ends[0];
            stg.plan(off, (size_t)(nrows + 1) * 8);
            if (str_nbytes[k])
                stg.plan(static_cast<const unsigned char *>(aggs[k].order) + ends[0], (size_t)str_nbytes[k]);
            if (aggs[k].mask)
                stg.plan(aggs[k].mask, (size_t)nrows);
            continue;
        }
        if (aggs[k].data)
            stg.plan(aggs[k].data, (size_t)nrows * dtype_size(a->dtype));
        if (aggs[k].order)
            stg.plan(aggs[k].order, a->op == B200_AGG_NUNIQUE ? (size_t)nrows : (size_t)nrows * dtype_size(a->dtype2));
        if (aggs[k].mask) {
            const bool first = a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST;
            stg.plan(aggs[k].mask, first ? (size_t)std::min<int64_t>(nrows, 1024) : (size_t)nrows);
        }
    }
    B200_CHECK(stg.commit());
    bool vec = true;
    auto chk = [&](const void *p) {
        if (p && (reinterpret_cast<uintptr_t>(p) & 15))
            vec = false;
    };
    for (int i = 0; i < nbinners; i++) {
        db[i].data = stg.dev(binners[i].data);
        db[i].mask = static_cast<const uint8_t *>(stg.dev(binners[i].mask));
        chk(db[i].data);
        chk(db[i].mask);
    }

    // split the aggregators: count/sum/min/max fuse into launches of <= B200_MAX_AGGS; first/last run their two passes each
    BinParams p;
    memset(&p, 0, sizeof p);
    p.nb = nbinners;
    p.nrows = nrows;
    p.cells = cells;
    memcpy(p.b, db, sizeof(DevBinner) * nbinners);
    auto flush = [&]() -> int {
        if (!p.na)
            return B200_OK;
        bool v = vec;
        for (int k = 0; k < p.na; k++) {
            if (p.a[k].data && (reinterpret_cast<uintptr_t>(p.a[k].data) & 15))
                v = false;
            if (p.a[k].mask && (reinterpret_cast<uintptr_t>(p.a[k].mask) & 15))
                v = false;
        }
        // privatise in shared memory when one copy of every grid fits comfortably (several copies for tiny grids)
        size_t copy = 0;
        for (int k = 0; k < p.na; k++) {
            p.a[k].smem_cell = p.a[k].op == B200_AGG_COUNT ? 4 : dtype_size(p.a[k].cell_dtype);
            copy = align_up(copy, 16);
            p.a[k].smem_off = (int)copy;
            copy += (size_t)cells * p.a[k].smem_cell;
        }
        copy = align_up(copy, 16);
        const size_t budget = 96 * 1024;
        p.smem_copies = 0;
        p.smem_copy_bytes = (int)copy;
        if (copy <= budget && nrows >= 4096) {
            int copies = (int)std::min<size_t>(8, (32 * 1024) / copy);
            p.smem_copies = copies < 1 ? 1 : copies;
        }
        int rc = launch_binby(ctx, sl, p, v);
        p.na = 0;
        return rc;
    };
    for (int k = 0; k < naggs; k++) {
        b200_agg *a = aggs[k].agg;
        if (a->op == B200_AGG_FIRST || a->op == B200_AGG_LAST) {
            FirstParams fp;
            memset(&fp, 0, sizeof fp);
            fp.nb = nbinners;
            fp.nrows = nrows;
            fp.row_offset = row_offset;
            memcpy(fp.b, db, sizeof(DevBinner) * nbinners);
            fp.dtype = a->dtype;
            fp.isz = dtype_size(a->dtype);
            fp.dtype2 = a->dtype2;
            fp.isz2 = dtype_size(a->dtype2);
            fp.byteswap = a->byteswap;
            fp.invert = a->op == B200_AGG_LAST;
            fp.data = stg.dev(aggs[k].data);
            fp.order = stg.dev(aggs[k].order);
            fp.mask = static_cast<const uint8_t *>(stg.dev(aggs[k].mask));
            fp.grid = a->grid;
            fp.order_grid = a->order;
            fp.state = static_cast<unsigned long long *>(a->state);
            fp.cell_masked = a->cell_masked;
            bool v = vec && !(reinterpret_cast<uintptr_t>(fp.data) & 15) && !(reinterpret_cast<uintptr_t>(fp.order) & 15);
            // select+deposit of one aggregator must not interleave with another slot's pair on the same grid: pairs are chained
            // through an event (stream-ordered across slots, no host or device-wide synchronisation)
            {
                std::lock_guard<std::mutex> chain(a->chain_mu);
                B200_CUDA(cudaStreamWaitEvent(st, a->chain, 0));
                B200_CHECK(launch_first(ctx, st, fp, v));
                B200_CUDA(cudaEventRecord(a->chain, st));
            }
            continue;
        }
        if (a->op == B200_AGG_LIST) {
            B200_CHECK(bin_list(ctx, sl, a, db, nbinners, stg.dev(aggs[k].data), static_cast<const uint8_t *>(stg.dev(aggs[k].mask)), nrows, vec));
            continue;
        }
        if (a->op == B200_AGG_LIST_STRING) {
            const unsigned char *bytes = str_nbytes[k] ? static_cast<const unsigned char *>(stg.dev(static_cast<const unsigned char *>(aggs[k].order) + str_first[k])) : nullptr;
            B200_CHECK(bin_list_string(sl, a, db, nbinners, static_cast<const long long *>(stg.dev(aggs[k].data)), bytes, str_first[k], (unsigned long long)str_nbytes[k],
                                       static_cast<const uint8_t *>(stg.dev(aggs[k].mask)), nrows, vec));
            continue;
        }
        if (a->op == B200_AGG_NUNIQUE) {
            B200_CHECK(bin_nunique(ctx, sl, a, db, nbinners, stg.dev(aggs[k].data), static_cast<const uint8_t *>(stg.dev(aggs[k].mask)),
                                   static_cast<const uint8_t *>(stg.dev(aggs[k].order)), nrows, vec));
            continue;
        }
        DevAgg &d = p.a[p.na++];
        memset(&d, 0, sizeof d);
        d.op = a->op;
        d.dtype = a->dtype;
        d.isz = dtype_size(a->dtype);
        d.byteswap = a->byteswap && d.isz > 1;
        d.cell_dtype = a->cell_dtype;
        d.moment = a->moment;
        d.init_bits = agg_init_bits(a->op, a->cell_dtype);
        d.data = stg.dev(aggs[k].data);
        d.mask = static_cast<const uint8_t *>(stg.dev(aggs[k].mask));
        d.grid = a->grid;
        if (p.na == B200_MAX_AGGS)
            B200_CHECK(flush());
    }
    B200_CHECK(flush());

    if (memspace == B200_MEM_MIXED && !(flags & B200_FLAG_ASYNC_HOST)) {
        // MIXED copies straight from the caller's host buffers, which are only valid during the call (vaex/cpu.py:708-710).
        // Plain HOST chunks were memcpy'd into the slot's page-locked bounce ring: nothing of the caller's is read after return,
        // so there is no wait here and the next chunk (another slot, or this one) overlaps this chunk's copy and kernels.
        B200_CUDA(cudaStreamSynchronize(st));
    }
    return B200_OK;
}

} // extern "C"

