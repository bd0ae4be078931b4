// ntt_fast_fq.cu -- fused negacyclic products for small moduli with FLOAT-QUOTIENT arithmetic
// (fq_arith.cuh): every twiddle product is one FFMA (quotient, read straight out of the mantissa) plus two
// low-half IMADs (remainder).  No IMAD.HI, no shifts, no int<->float conversions, no range compressions:
// values travel biased by 0x4B400000 so that the same register is an integer for the IMADs and the float
// 1.5 * 2^23 + x for the FFMA.  Per butterfly: FFMA + 2 IMAD + 2 IADD3 = 5 issue slots spread over the
// fma-lite, fma-heavy and ALU pipes (measured 5.6e12 butterflies/s against 3.9e12 for the IMAD/IMAD.HI/IMAD
// Barrett butterfly of ntt_fast_sq.cu, profiles/int_peaks_r02.txt).
//
// This file: the arithmetic on the r01 schedule of fast_common.cuh (n/8 threads per polynomial, 8 coefficients
// per thread, three radix-2 stages per register pass, shared-memory tile between passes, both operands of a
// product share a pass's twiddle registers).  It is the SCGPU_FAST_ARITH=3 cross-check; production products go
// through the warp-local 32-coefficient schedule (warp32.cuh, ntt_fast_fq32.cu).  Twiddles: two parallel arrays
// (w, wq), k and c rebuilt per entry; pass-0 entries from the constant bank.
//
// Exactness: the host proves by interval propagation over this dataflow (fq_host.h: analyse) that every
// value read as a float stays below 2^22 and that the last product lies in (-q, q); tools/fq_model.cpp runs
// the same arithmetic on the CPU against a schoolbook product.  Inputs beyond +-4q (never passed by a scheme)
// are detected by a warp vote and reduced first, so any SINT32 input is exact.
#include "scgpu_internal.h"
#include "fast_common.cuh"
#include "fq_host.h"
#include "../../include/scgpu.h"

#include <algorithm>
#include <vector>

namespace scgpu {

using namespace fast;

namespace {

using fq::Tw;
using fq::kBias;

// Twiddle tables are stored as two parallel arrays (w[n], wq[n]) so that a thread's 4 (2, 1) consecutive
// entries of a stage are ONE 128 (64, 32)-bit load and a warp's loads are contiguous: 16-byte {w,wq,k,c}
// records cost 408 L1 tag requests per product and made the first version of this kernel LSU-bound
// (profiles/polymul_r02a_*).  k and c are rebuilt with one IMAD and one FFMA per entry.  The entries of
// pass 0 are the same for every thread and come from the kernel's constant bank instead.
struct FqTab { const int32_t *w; const float *wq; };

struct FqConst {
    FqTab zf;               // [n] psi^brv(k)
    FqTab zi;               // [n] inverses; entry 1 carries n^-1 and is unbiased
    Tw f0[7], i0[7];        // pass-0 entries (stage s, block 0..2^s-1 at index 2^s - 1 + b), forward / inverse
    Tw ninv;                // n^-1, unbiased result (sum branch of the last inverse stage)
    Tw one;                 // multiplication by 1 = reduction, biased result
    int32_t q, nq, x0, pwk; // nq = -q; pwk = kBias * q
    int32_t kf, ki;         // k = w * (-kBias) + kf (forward, unbiased result) / + ki (inverse, biased result)
    float invq;
    uint32_t M;             // floor(2^32 / q): 32-bit Barrett of the out-of-range path
    int r_inv[4];
};

typedef uint32_t u32;

__device__ __forceinline__ Tw derive(int32_t w, int32_t wqbits, int32_t kbase)
{
    Tw t;
    t.w = w;
    t.wq = __int_as_float(wqbits);
    t.k = fq::mad(w, -kBias, kbase);
    t.c = __fmaf_rn(t.wq, -fq::kBiasF, fq::kBiasF);        // 1.5 * 2^23 - 3 * k22, exact
    return t;
}

// exact residue of any 32-bit value, |result| < q (only on the out-of-range path)
__device__ __forceinline__ int32_t bred(int32_t p, const FqConst &c)
{
    const int32_t qe = (int32_t)(((int64_t)p * (int64_t)c.M + 0x80000000ll) >> 32);
    return qe * c.nq + p;
}

struct FqTw { Tw z4; Tw z2[2]; Tw z1[4]; };

template <int LOGN, int PASS, bool INV>
__device__ __forceinline__ void fq_load_tw(FqTw &tw, const FqConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    if (PASS == 0) {
        // C::J == 3, block 0: entries 1, 2..3, 4..7 of the table
        const Tw *t0 = INV ? c.i0 : c.f0;
        tw.z4 = t0[0];
        tw.z2[0] = t0[1]; tw.z2[1] = t0[2];
#pragma unroll
        for (int i = 0; i < 4; i++) tw.z1[i] = t0[3 + i];
        return;
    }
    const FqTab &zt = INV ? c.zi : c.zf;
    const int32_t kb = INV ? c.ki : c.kf;
    const int blk = tau / C::D;
    if (C::J == 3) {
        const int i = (1 << C::S0) + blk;
        tw.z4 = derive(__ldg(zt.w + i), __float_as_int(__ldg(zt.wq + i)), kb);
    }
    if (C::J >= 2) {
        const int i = (1 << (C::S0 + C::J - 2)) + 2 * blk;
        const int2 w = __ldg(reinterpret_cast<const int2 *>(zt.w + i));
        const int2 f = __ldg(reinterpret_cast<const int2 *>(zt.wq + i));
        tw.z2[0] = derive(w.x, f.x, kb);
        tw.z2[1] = derive(w.y, f.y, kb);
    }
    {
        const int i = (1 << (C::S0 + C::J - 1)) + 4 * blk;
        const int4 w = __ldg(reinterpret_cast<const int4 *>(zt.w + i));
        const int4 f = __ldg(reinterpret_cast<const int4 *>(zt.wq + i));
        tw.z1[0] = derive(w.x, f.x, kb);
        tw.z1[1] = derive(w.y, f.y, kb);
        tw.z1[2] = derive(w.z, f.z, kb);
        tw.z1[3] = derive(w.w, f.w, kb);
    }
}

// all coefficients are biased (x + kBias) and kept in unsigned registers: sums wrap, never overflow
__device__ __forceinline__ void fq_ct(u32 &lo, u32 &hi, const Tw &z, int32_t nq)
{
    const u32 t = (u32)fq::mul((int32_t)hi, z, nq);
    hi = lo - t;
    lo = lo + t;
}
__device__ __forceinline__ void fq_gs(u32 &lo, u32 &hi, const Tw &z, int32_t nq)
{
    const u32 d = lo - hi + (u32)kBias;
    lo = lo + hi - (u32)kBias;
    hi = (u32)fq::mul((int32_t)d, z, nq);          // z.k carries the bias of the result
}

template <int J>
__device__ __forceinline__ void fq_fwd_pass(u32 (&x)[8], const FqTw &tw, int32_t nq)
{
    if (J == 3) {
#pragma unroll
        for (int m = 0; m < 4; m++) fq_ct(x[m], x[m + 4], tw.z4, nq);
    }
    if (J >= 2) {
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) fq_ct(x[m], x[m + 2], tw.z2[m >> 2], nq);
    }
#pragma unroll
    for (int m = 0; m < 8; m += 2) fq_ct(x[m], x[m + 1], tw.z1[m >> 1], nq);
}

template <int LOGN, int PASS>
__device__ __forceinline__ void fq_tile_store(int32_t *tile, const u32 (&x)[8], int tau)
{
#pragma unroll
    for (int m = 0; m < 8; m++) tile[swz<LOGN>(elem_index<PassCfg<LOGN, PASS>::D>(tau, m))] = (int32_t)x[m];
}
template <int LOGN, int PASS>
__device__ __forceinline__ void fq_tile_load(const int32_t *tile, u32 (&x)[8], int tau)
{
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = (u32)tile[swz<LOGN>(elem_index<PassCfg<LOGN, PASS>::D>(tau, m))];
}

template <int LOGN, int PASS, int NOPS>
__device__ __forceinline__ void fq_fwd_all(u32 (&xa)[8], u32 (&xb)[8], int32_t *ta, int32_t *tb,
                                           const FqConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    FqTw tw;
    fq_load_tw<LOGN, PASS, false>(tw, c, tau);
    if (PASS > 0) {
        group_sync<LOGN>();
        fq_tile_load<LOGN, PASS>(ta, xa, tau);
        if (NOPS == 2) fq_tile_load<LOGN, PASS>(tb, xb, tau);
    }
    fq_fwd_pass<C::J>(xa, tw, c.nq);
    if (NOPS == 2) fq_fwd_pass<C::J>(xb, tw, c.nq);
    if constexpr (PASS + 1 < NumPasses<LOGN>::value) {
        fq_tile_store<LOGN, PASS>(ta, xa, tau);
        if (NOPS == 2) fq_tile_store<LOGN, PASS>(tb, xb, tau);
        fq_fwd_all<LOGN, PASS + 1, NOPS>(xa, xb, ta, tb, c, tau);
    }
}

// x: biased on entry; canonical residues in [0, q) on return
template <int LOGN, int PASS>
__device__ __forceinline__ void fq_inv_all(u32 (&x)[8], int32_t *tile, const FqConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    FqTw tw;
    fq_load_tw<LOGN, PASS, true>(tw, c, tau);
    if (PASS + 1 < NumPasses<LOGN>::value) {
        group_sync<LOGN>();
        fq_tile_load<LOGN, PASS>(tile, x, tau);
    }
    if (c.r_inv[PASS]) {
#pragma unroll
        for (int m = 0; m < 8; m++) x[m] = (u32)fq::mul((int32_t)x[m], c.one, c.nq);
    }
#pragma unroll
    for (int m = 0; m < 8; m += 2) fq_gs(x[m], x[m + 1], tw.z1[m >> 1], c.nq);
    if (C::J >= 2) {
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) fq_gs(x[m], x[m + 2], tw.z2[m >> 2], c.nq);
    }
    if constexpr (PASS == 0) {
        // stage 0: both branches are multiplied (n^-1 on the sum, n^-1 * zeta^-1 on the difference); both
        // products are unbiased and proven to lie in (-q, q): one conditional +q gives the canonical residue
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const u32 s = x[m] + x[m + 4] - (u32)kBias;
            const u32 d = x[m] - x[m + 4] + (u32)kBias;
            const u32 ys = (u32)fq::mul((int32_t)s, c.ninv, c.nq);
            const u32 yd = (u32)fq::mul((int32_t)d, tw.z4, c.nq);
            x[m] = min(ys, ys + (u32)c.q);
            x[m + 4] = min(yd, yd + (u32)c.q);
        }
    } else {
        if (C::J == 3) {
#pragma unroll
            for (int m = 0; m < 4; m++) fq_gs(x[m], x[m + 4], tw.z4, c.nq);
        }
        fq_tile_store<LOGN, PASS>(tile, x, tau);
        fq_inv_all<LOGN, PASS - 1>(x, tile, c, tau);
    }
}

// raw SINT32 -> in range; `wide` accumulates "some |x| > x0" for the caller's warp vote
__device__ __forceinline__ bool out_of_range(int32_t v, const FqConst &c)
{
    return ((u32)v + (u32)c.x0) > (u32)(2 * c.x0);
}

template <int LOGN>
__device__ __forceinline__ void fq_load_operand(u32 (&x)[8], const int32_t *row, int tau, const FqConst &c)
{
    constexpr int D0 = PassCfg<LOGN, 0>::D;
    int32_t v[8];
    bool wide = false;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        v[m] = __ldg(row + tau + m * D0);
        wide |= out_of_range(v[m], c);
    }
    if (__any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
        for (int m = 0; m < 8; m++) v[m] = bred(v[m], c);
    }
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = (u32)v[m] + (u32)kBias;
}

enum { FQ_POLYMUL = 0, FQ_KEY16 = 1, FQ_KEY32 = 2 };

template <int LOGN, int MODE>
__global__ void __launch_bounds__(kCtaThreads, 3)
k_polymul_fq(int32_t *__restrict__ out, const int32_t *__restrict__ a, const void *__restrict__ bsrc,
             size_t b_stride, size_t count, const __grid_constant__ FqConst c)
{
    constexpr int N = 1 << LOGN;
    constexpr int T = N / 8;
    constexpr int G = kCtaThreads / T;
    constexpr int D0 = PassCfg<LOGN, 0>::D;
    constexpr int LAST = NumPasses<LOGN>::value - 1;
    __shared__ __align__(16) int32_t tiles[2][G][N];
    const int g = threadIdx.x / T;
    const int tau = threadIdx.x % T;
    int32_t *ta = tiles[0][g];
    int32_t *tb = tiles[1][g];

    for (size_t base = (size_t)blockIdx.x * G; base < count; base += (size_t)gridDim.x * G) {
        const size_t poly = base + g;
        const bool live = poly < count;
        const size_t prow = live ? poly : 0;
        u32 xa[8], xb[8];
        fq_load_operand<LOGN>(xa, a + prow * N, tau, c);
        if (MODE == FQ_POLYMUL) {
            fq_load_operand<LOGN>(xb, static_cast<const int32_t *>(bsrc) + prow * b_stride, tau, c);
            fq_fwd_all<LOGN, 0, 2>(xa, xb, ta, tb, c, tau);
#pragma unroll
            for (int m = 0; m < 8; m++)
                xa[m] = (u32)fq::mul_var((int32_t)(xa[m] - (u32)kBias), (int32_t)(xb[m] - (u32)kBias), c.invq, c.pwk, c.nq) + (u32)kBias;
        } else {
            fq_fwd_all<LOGN, 0, 1>(xa, xb, ta, tb, c, tau);
            int32_t kv[8];
            bool wide = false;
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int j = (int)(__brev((unsigned)(elem_index<PassCfg<LOGN, LAST>::D>(tau, m))) >> (32 - LOGN));
                if (MODE == FQ_KEY16) kv[m] = (int32_t)__ldg(static_cast<const int16_t *>(bsrc) + prow * b_stride + j);
                else {
                    kv[m] = __ldg(static_cast<const int32_t *>(bsrc) + prow * b_stride + j);
                    wide |= out_of_range(kv[m], c);
                }
            }
            if (MODE == FQ_KEY32 && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                for (int m = 0; m < 8; m++) kv[m] = bred(kv[m], c);
            }
#pragma unroll
            for (int m = 0; m < 8; m++)
                xa[m] = (u32)fq::mul_var((int32_t)(xa[m] - (u32)kBias), kv[m], c.invq, c.pwk, c.nq) + (u32)kBias;
        }
        fq_inv_all<LOGN, LAST>(xa, ta, c, tau);
        if (live) {
            int32_t *orow = out + poly * N;
#pragma unroll
            for (int m = 0; m < 8; m++) orow[tau + m * D0] = (int32_t)xa[m];
        }
        group_sync<LOGN>();
    }
}

// module-LWE matrix-vector product t_i = INTT(sum_j A_ij o NTT(s_j)), same structure as k_matvec (ntt_fast.cu)
// SHARED_A: one matrix for every instance (instance stride 0)
template <int LOGN, int MAXL, bool SHARED_A = false>
__global__ void __launch_bounds__(kCtaThreads)
k_matvec_fq(int32_t *__restrict__ out, const int32_t *__restrict__ A, const int32_t *__restrict__ s,
            int k, int l, size_t count, const __grid_constant__ FqConst c)
{
    constexpr int N = 1 << LOGN;
    constexpr int T = N / 8;
    constexpr int G = kCtaThreads / T;
    constexpr int D0 = PassCfg<LOGN, 0>::D;
    constexpr int LAST = NumPasses<LOGN>::value - 1;
    __shared__ __align__(16) int32_t tiles[G][N];
    __shared__ __align__(16) int32_t stash[G][MAXL][N];
    const int g = threadIdx.x / T;
    const int tau = threadIdx.x % T;
    int32_t *tile = tiles[g];
    for (size_t base = (size_t)blockIdx.x * G; base < count; base += (size_t)gridDim.x * G) {
        const size_t inst = base + g;
        const bool live = inst < count;
        const size_t irow = live ? inst : 0;
        u32 dummy[8];
        for (int j = 0; j < l; j++) {
            u32 x[8];
            fq_load_operand<LOGN>(x, s + (irow * l + j) * N, tau, c);
            fq_fwd_all<LOGN, 0, 1>(x, dummy, tile, tile, c, tau);
#pragma unroll
            for (int m = 0; m < 8; m++) stash[g][j][m * T + tau] = (int32_t)(x[m] - (u32)kBias);     // |.| <= forward bound
            group_sync<LOGN>();
        }
        for (int i = 0; i < k; i++) {
            u32 acc[8];
#pragma unroll
            for (int m = 0; m < 8; m++) acc[m] = (u32)kBias;
            for (int j = 0; j < l; j++) {
                const int32_t *arow = A + (((SHARED_A ? (size_t)0 : irow * k) + i) * l + j) * N;
                int32_t av[8];
                bool wide = false;
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    const int idx = (int)(__brev((unsigned)(elem_index<PassCfg<LOGN, LAST>::D>(tau, m))) >> (32 - LOGN));
                    av[m] = __ldg(arow + idx);
                    wide |= out_of_range(av[m], c);
                }
                // A is canonical in the reference (sampled in [0, q)); anything else is reduced first
                if (__any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                    for (int m = 0; m < 8; m++) av[m] = bred(av[m], c);
                }
#pragma unroll
                for (int m = 0; m < 8; m++)
                    acc[m] += (u32)fq::mul_var(av[m], stash[g][j][m * T + tau], c.invq, c.pwk, c.nq);
            }
            fq_inv_all<LOGN, LAST>(acc, tile, c, tau);
            if (live) {
                int32_t *orow = out + (inst * k + i) * N;
#pragma unroll
                for (int m = 0; m < 8; m++) orow[tau + m * D0] = (int32_t)acc[m];
            }
            group_sync<LOGN>();
        }
    }
}

}  // namespace

struct FqState {
    int32_t *zf, *zi;       // w[n] followed by wq[n]
    FqConst prod, mv;       // mv: range reductions for up to 4 accumulated products
};

int build_fq_tables(NttPlanDev &p, const int32_t *w_host)
{
    if (p.logn < 8 || p.logn > 10) return SCGPU_OK;
    const fq::Schedule s1 = fq::analyse(p.logn, p.rc.q, 1);
    const fq::Schedule s4 = fq::analyse(p.logn, p.rc.q, 4);
    if (!s1.ok || !s4.ok) return SCGPU_OK;                 // the Barrett / Montgomery kernels serve this (q, n)
    std::vector<Tw> zf, zi;
    FqConst c;
    if (!fq::build_tables(p.logn, p.rc.q, w_host, zf, zi, c.ninv, c.one)) return SCGPU_OK;
    // device tables: w[n] followed by wq[n]; the derived k / c of every entry equal the host-built ones
    // (checked here so that a table the derivation cannot reproduce is never used)
    std::vector<int32_t> packf(2 * p.n), packi(2 * p.n);
    const int32_t pwk = (int32_t)((uint32_t)kBias * (uint32_t)p.rc.q);
    for (int k = 0; k < p.n; k++) {
        packf[k] = zf[k].w; memcpy(&packf[p.n + k], &zf[k].wq, 4);
        packi[k] = zi[k].w; memcpy(&packi[p.n + k], &zi[k].wq, 4);
        const int32_t kf = fq::mad(zf[k].w, -kBias, pwk);
        const int32_t ki = fq::mad(zi[k].w, -kBias, (int32_t)((uint32_t)pwk + (uint32_t)kBias));
        const bool okf = kf == zf[k].k && fmaf(zf[k].wq, -fq::kBiasF, fq::kBiasF) == zf[k].c;
        const bool oki = (k < 2 || ki == zi[k].k) && fmaf(zi[k].wq, -fq::kBiasF, fq::kBiasF) == zi[k].c;
        if (!okf || !oki) { set_error("float-quotient table self-check failed at entry %d", k); return SCGPU_ERR_ARG; }
    }
    FqState *s = p.fq = new FqState();
    SCGPU_CUDA_CHECK(cudaMalloc(&s->zf, sizeof(int32_t) * 2 * p.n));
    SCGPU_CUDA_CHECK(cudaMalloc(&s->zi, sizeof(int32_t) * 2 * p.n));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->zf, packf.data(), sizeof(int32_t) * 2 * p.n, cudaMemcpyHostToDevice));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->zi, packi.data(), sizeof(int32_t) * 2 * p.n, cudaMemcpyHostToDevice));
    c.zf.w = s->zf;
    c.zf.wq = reinterpret_cast<const float *>(s->zf + p.n);
    c.zi.w = s->zi;
    c.zi.wq = reinterpret_cast<const float *>(s->zi + p.n);
    std::copy(zf.begin() + 1, zf.begin() + 8, c.f0);         // pass 0: entries 1..7
    std::copy(zi.begin() + 1, zi.begin() + 8, c.i0);
    c.q = p.rc.q; c.nq = -p.rc.q; c.x0 = s1.x0;
    c.pwk = pwk;
    c.kf = c.pwk;
    c.ki = (int32_t)((uint32_t)c.pwk + (uint32_t)kBias);
    c.invq = (float)(1.0 / (double)p.rc.q);
    c.M = (uint32_t)((1ull << 32) / (uint64_t)p.rc.q);
    s->prod = s->mv = c;
    for (int i = 0; i < 4; i++) { s->prod.r_inv[i] = s1.r_inv[i]; s->mv.r_inv[i] = s4.r_inv[i]; }
    return SCGPU_OK;
}

void free_fq_tables(NttPlanDev &p)
{
    if (!p.fq) return;
    cudaFree(p.fq->zf);
    cudaFree(p.fq->zi);
    delete p.fq;
    p.fq = nullptr;
}

int launch_polymul_fq(const NttPlanDev &p, int mode, int32_t *out, const int32_t *a, const void *b,
                      size_t b_stride, size_t count, cudaStream_t st)
{
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 3);
    return with_int<8, 9, 10>(p.logn, [&](auto L) {
        return with_int<FQ_POLYMUL, FQ_KEY16, FQ_KEY32>(mode, [&](auto M) {
            return launch_kernel(k_polymul_fq<L, M>, grid, kCtaThreads, 0, st, out, a, b, b_stride, count, p.fq->prod);
        });
    });
}

int launch_matvec_fq(const NttPlanDev &p, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                     size_t count, cudaStream_t st, bool shared)
{
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 2);
    if (shared) return launch_kernel(k_matvec_fq<8, 4, true>, grid, kCtaThreads, 0, st, out, A, s, k, l, count, p.fq->mv);
    return launch_kernel(k_matvec_fq<8, 4>, grid, kCtaThreads, 0, st, out, A, s, k, l, count, p.fq->mv);
}

}  // namespace scgpu
