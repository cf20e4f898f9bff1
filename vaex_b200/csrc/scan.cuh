// scan.cuh — exclusive scan of u32 / u64 counters in place, one CTA (shared by the radix sort of hashset.cu, the filter compaction
// of expr.cu and the list finalisation of list.cu: n is a few million at most).
#pragma once
#include "common.cuh"

namespace b200 {

// total (optional) receives the sum of all counters
template <class T>
static __device__ __forceinline__ void scan_excl_cta(T *a, unsigned long long n, unsigned long long *total) {
    __shared__ T warp_sums[32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0)
        carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (unsigned long long base = 0; base < n; base += 1024) {
        const unsigned long long i = base + threadIdx.x;
        const T v = i < n ? a[i] : T(0);
        T x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o)
                x += y;
        }
        if (lane == 31)
            warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            T w = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const T y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o)
                    w += y;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const unsigned long long before = carry + (warp ? warp_sums[warp - 1] : T(0)) + x - v;
        if (i < n)
            a[i] = (T)before;
        __syncthreads();
        if (threadIdx.x == 1023)
            carry = before + v;
        __syncthreads();
    }
    if (total && threadIdx.x == 0)
        *total = carry;
}

static __global__ void __launch_bounds__(1024) k_scan_u32(unsigned *a, unsigned long long n, unsigned long long *total = nullptr) { scan_excl_cta(a, n, total); }
static __global__ void __launch_bounds__(1024) k_scan_u64(unsigned long long *a, unsigned long long n, unsigned long long *total = nullptr) {
    scan_excl_cta(a, n, total);
}

} // namespace b200
