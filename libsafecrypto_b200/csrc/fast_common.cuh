// fast_common.cuh -- register-pass schedule shared by the fused kernels (ntt_fast.cu: Montgomery,
// any odd q < 2^30; ntt_fast_sq.cu: 32-bit Barrett for small q).
//
// n/8 threads per polynomial, 8 coefficients ("slots") per thread.  Pass p covers radix-2 stages
// [3p, 3p+J) with slot stride D: thread tau holds elements (tau / D) * 8D + tau % D + m * D, m = 0..7, so a
// stage whose butterfly distance is delta * D pairs slots (m, m + delta).  Between passes coefficients go
// through a shared-memory tile whose index is XOR-swizzled so that every pass's access pattern (fixed m,
// 32 lanes) hits 32 distinct banks (tests/test_layout.py).
#pragma once
#include <cstdint>

namespace scgpu {
namespace fast {

constexpr int kCtaThreads = 256;

template <int LOGN>
__device__ __forceinline__ int swz(int idx)
{
    if (LOGN == 8)  return idx ^ ((idx >> 5) & 7) ^ (((idx >> 5) & 3) << 3);
    if (LOGN == 9)  return idx ^ ((idx >> 5) & 7) ^ (((idx >> 6) & 3) << 3);
    return idx ^ ((idx >> 5) & 7) ^ (((idx >> 5) & 1) << 3) ^ (((idx >> 7) & 1) << 4);
}

// pass p of the schedule: stages [3p, 3p + J), slot stride D
template <int LOGN, int PASS>
struct PassCfg {
    static constexpr int N = 1 << LOGN;
    static constexpr int S0 = 3 * PASS;
    static constexpr int J = (LOGN - S0) >= 3 ? 3 : (LOGN - S0);
    static constexpr int D = (J == 3) ? (N >> (S0 + 3)) : 1;
};
template <int LOGN> struct NumPasses { static constexpr int value = (LOGN + 2) / 3; };

template <int D>
__device__ __forceinline__ int elem_index(int tau, int m)
{
    return (tau / D) * (8 * D) + (tau % D) + m * D;
}

// Barrier over the n/8 threads that share one polynomial's tile (not the whole CTA): a warp-level sync for
// n = 256, a named barrier (ids 1..) for n = 512 / 1024.  Polynomials in a CTA never wait for each other.
template <int LOGN>
__device__ __forceinline__ void group_sync()
{
    constexpr int T = (1 << LOGN) / 8;
    if (T == 32) {
        __syncwarp();
    } else {
        const int id = 1 + (int)threadIdx.x / T;
        asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(T) : "memory");
    }
}

template <int LOGN, int PASS>
__device__ __forceinline__ void tile_store(int32_t *tile, const int32_t (&x)[8], int tau)
{
#pragma unroll
    for (int m = 0; m < 8; m++) tile[swz<LOGN>(elem_index<PassCfg<LOGN, PASS>::D>(tau, m))] = x[m];
}
template <int LOGN, int PASS>
__device__ __forceinline__ void tile_load(const int32_t *tile, int32_t (&x)[8], int tau)
{
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = tile[swz<LOGN>(elem_index<PassCfg<LOGN, PASS>::D>(tau, m))];
}

// grid-stride launch of `count` polynomials (n/8 threads each): per_sm resident CTAs per SM, no more CTAs than groups
inline unsigned cta_grid(int sm_count, int n, size_t count, int per_sm)
{
    const size_t G = kCtaThreads / (n / 8), groups = (count + G - 1) / G;
    size_t grid = (size_t)(sm_count > 0 ? sm_count : 148) * per_sm;
    if (grid > groups) grid = groups;
    return grid == 0 ? 1u : (unsigned)grid;
}

}  // namespace fast
}  // namespace scgpu
