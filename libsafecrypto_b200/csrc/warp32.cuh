// warp32.cuh -- the warp-local 32-coefficient schedule of the fused kernels, generic in the modular arithmetic:
// W32<AR> holds the device code (passes, exchanges, operand loading), k_polymul_w32 / k_matvec_w32 are the
// kernels; AR is an arithmetic policy (ArFq: float-quotient products for small moduli, ntt_fast_fq32.cu;
// ArSh: Shoup products + Montgomery pointwise for moduli up to 2^26, ntt_fast_sh32.cu).  See ntt_fast_fq32.cu
// for the description of the schedule.
//
// Policy interface:  E (twiddle entry), K (scalar constants), WORDS (32-bit words of E in the tables),
//   enc / dec / zero            raw <-> internal representation of a coefficient, internal zero
//   cb(e)                       entry read from the kernel's constant bank
//   PASS0_IMM                   true: AR::fwd_pass0(x, k) / AR::inv_pass0(x, k) replace the table-driven pass 0 (entries
//                               compiled into the policy); serves<LOGN, MODE, BM>() limits the kernels it is built for
//   mk(words)                   entry from WORDS table words
//   ct / gs                     forward / inverse butterfly on internal values
//   ct0                         ct whose lo operand is still RAW (stage 0 encodes it for free in its 3-input adds)
//   fin(lo, hi, ninv, z, k)     last inverse stage: both branches scaled, canonical residues out
//   red(x, one, k)              x * 1 mod q (range reduction), internal in / out
//   pw(a, b, k)                 pointwise product of two internal values, internal out
//   pwraw(a, kv, k)             internal a times raw kv, internal out
//   Acc, acc_zero / acc_add(acc, av, sv, k) / acc_fin(acc, k)
//                               accumulator of raw av times decoded sv over the mat-vec's inner index; acc_fin
//                               returns the internal representation of the sum
#pragma once
#include "scgpu_internal.h"
#include "../../include/scgpu.h"

#include <cstdint>
#include <cstdlib>

namespace scgpu {
namespace w32 {

typedef uint32_t u32;



#ifndef W32_THREADS
#define W32_THREADS 32
#endif
// one warp per CTA: warps never synchronise with each other, and 20 independent one-warp CTAs per SM measured
// 2-3 % faster than 5 CTAs of 4 warps (finer-grained scheduling at the tail, no co-scheduling of a CTA's warps)
constexpr int kThreads32 = W32_THREADS;
#ifndef FQ32_MINB
#define FQ32_MINB 20
#endif

template <int LOGN>
struct Cfg32 {
    static constexpr int N = 1 << LOGN;
    static constexpr int T = N / 32;             // threads per polynomial
    static constexpr int PW = 32 / T;            // polynomials per warp
    static constexpr int SUB = N / 32 > 16 ? 16 : N / 32;   // elements of one pass-1 sub-chunk
    static constexpr int NSUB = 32 / SUB;
    // first stage of the sub-chunk loop.  n = 1024: stage 5 couples all 32 elements of a thread; it runs as a
    // separate step over the whole chunk (one operand at a time) so that the sub-chunk loop holds 2 x 16
    // coefficients instead of 2 x 32 (168 -> 96 registers, 3 -> 5 CTAs per SM)
    static constexpr int S1 = LOGN == 10 ? 6 : 5;
    static constexpr int TS = N + N / 8 + (T & 31);   // tile stride in words (bank offset T between polynomials)
    static constexpr int POLYS = (kThreads32 / 32) * PW;
};

// padded tile position of element e
__host__ __device__ constexpr int pos32(int e) { return e + 4 * (e >> 5); }

template <int SUB>
__device__ __forceinline__ void load_sub(const int32_t *p, u32 (&x)[SUB])
{
#pragma unroll
    for (int k = 0; k < SUB; k += 4) {
        const int4 v = *reinterpret_cast<const int4 *>(p + k);
        x[k] = (u32)v.x; x[k + 1] = (u32)v.y; x[k + 2] = (u32)v.z; x[k + 3] = (u32)v.w;
    }
}
template <int SUB>
__device__ __forceinline__ void store_sub(int32_t *p, const u32 (&x)[SUB])
{
#pragma unroll
    for (int k = 0; k < SUB; k += 4)
        *reinterpret_cast<int4 *>(p + k) = make_int4((int32_t)x[k], (int32_t)x[k + 1], (int32_t)x[k + 2], (int32_t)x[k + 3]);
}

// ---- TMA bulk copies (cp.async.bulk) + mbarrier: the next product's operand rows are fetched into tile
// regions the current product no longer needs, by one lane per warp, while the warp computes ----------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int arrivals)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- dynamic work distribution -------------------------------------------------------------------------------
// The grids are persistent (one-warp CTAs, FQ32_MINB per SM).  With a static stride every warp owns the same number
// of groups, but the warps of a scheduler do not advance at the same rate: ncu showed 3.9 of 5 resident warps alive
// on average (profiles/polymul_r04_ncu.json), i.e. the favoured warps retire early and the last ones run alone.
// So the groups after the first grid-full are claimed from a global counter (zeroed by the launcher): lane 0 claims
// the NEXT group at the top of an iteration, which is when its rows are put in flight; the other lanes learn the
// index at the end of the iteration.  ctr == nullptr keeps the static stride (SCGPU_STATIC_SCHED=1).
static_assert(kThreads32 == 32, "the work counter is claimed per CTA: one warp per CTA");
// Group indices are 32-bit (one register across the iteration; the launchers refuse batches beyond 2^32 groups).
__device__ __forceinline__ unsigned claim_next(unsigned long long *ctr, unsigned g, int lane)
{
    if (ctr == nullptr) return g + gridDim.x;
    unsigned nxt = 0;
    if (lane == 0) nxt = atomicAdd(reinterpret_cast<unsigned *>(ctr), 1u) + gridDim.x;
    return nxt;                                             // meaningful on lane 0 only
}
__device__ __forceinline__ unsigned share_next(unsigned long long *ctr, unsigned gnext)
{
    return ctr == nullptr ? gnext : __shfl_sync(0xFFFFFFFFu, gnext, 0);
}
// Pipelined claim: a warp knows its current group g AND its next group gn (whose rows it prefetches); at the top of
// an iteration lane 0 claims the group AFTER the next one and nobody reads the atomic's result before the end of the
// iteration.  (Claiming the next group itself left the atomic's latency exposed wherever the prefetch is issued early
// in the iteration: the add that consumed its result was the most-sampled stall of the kernel,
// profiles/polymul_r2bm_ncu_mix.txt.)  The first two groups of a warp are static, the counter hands out the rest.
struct Claim {
    // Chunked claims: one atomic hands a warp kChunk consecutive groups while plenty of work is left, single groups near
    // the end.  With one atomic per group the canonical transforms asked one address for 0.7 atomics per ns (2^19 claims
    // in 0.75 ms, n = 512) -- about the rate at which an L2 slice serialises same-address atomics: depending on the
    // slot's slice the kernel ran at 0.87 or at 0.46 of HBM peak (profiles/ab_canonical_r2.txt).
    // The counter counts claims, every claim adds 1: claim c < nb is the chunk [2 grid + c kChunk, + kChunk), the later
    // ones are the single groups behind the chunks (the last 8 grid-fulls), so a claim's extent follows from its number.
    unsigned kChunk;                                         // groups per claim (1, 2 or 4: word 2 of the launch's slot)
    unsigned g, gn;                                          // current group, the group after it (prefetched)
    unsigned gend;                                           // end of the current chunk
    unsigned ns, nend;                                       // the next chunk
    unsigned raw, nb;                                        // claim in flight (lane 0); number of kChunk-sized claims
    unsigned *p;                                             // the counter, through an opaque per-lane register (see issue)
    __device__ __forceinline__ void init(unsigned long long *ctr, unsigned total)
    {
        g = blockIdx.x; gn = blockIdx.x + gridDim.x; raw = 0;
        gend = g + 1; ns = gn; nend = gn + 1;
        kChunk = ctr != nullptr ? reinterpret_cast<volatile unsigned *>(ctr)[2] : 1u;
        const unsigned reserve = 10u * gridDim.x;            // 2 static grid-fulls + 8 of single groups
        nb = (kChunk > 1u && total > reserve) ? (total - reserve) / kChunk : 0u;
        // ptxas turns an atomic add on a provably warp-uniform address into a warp-aggregated atomic -- leader election,
        // POPC, and a SHFL that broadcasts the result -- even when one lane issues it through inline PTX, and that shuffle
        // waits for the atomic on the spot (it was the most-sampled instruction of the kernel,
        // profiles/polymul_r2c_ncu_mix.txt).  An address that is not provably uniform keeps the atomic a plain one whose
        // result nobody reads before advance().
        // (the high word of the 64-bit slot is zero -- the launcher clears the slot and only the low word counts -- but
        // only at run time: the address below depends on a value each lane loaded for itself)
        p = reinterpret_cast<unsigned *>(ctr);
        if (ctr != nullptr) p += (threadIdx.x + 1u) * reinterpret_cast<volatile unsigned *>(ctr)[1];
    }
    // in the last group of a chunk: claim the chunk after the next one (read at the end of this iteration)
    __device__ __forceinline__ void issue(unsigned long long *ctr, int lane)
    {
        if (ctr != nullptr && lane == 0 && g + 1u == gend)
            asm volatile("atom.global.add.u32 %0, [%1], 1;" : "=r"(raw) : "l"(p) : "memory");
    }
    __device__ __forceinline__ void advance(unsigned long long *ctr)
    {
        if (ctr == nullptr) { g = gn; gn = gn + gridDim.x; return; }
        g++;
        if (g == gend) {
            unsigned c;
            asm volatile("shfl.sync.idx.b32 %0, %1, 0, 0x1f, 0xffffffff;" : "=r"(c) : "r"(raw) : "memory");
            g = ns; gend = nend;
            const unsigned base = 2u * gridDim.x;
            ns = c < nb ? base + c * kChunk : base + nb * kChunk + (c - nb);
            nend = ns + (c < nb ? kChunk : 1u);
        }
        gn = g + 1u < gend ? g + 1u : ns;
    }
};

template <int LOGN>
__device__ __forceinline__ void store_pass0(int32_t *tile, const u32 (&x)[32], int tau)
{
    constexpr int T = Cfg32<LOGN>::T;
#pragma unroll
    for (int m = 0; m < 32; m++) tile[tau + pos32(T * m)] = (int32_t)x[m];
}
template <int LOGN>
__device__ __forceinline__ void load_pass0(const int32_t *tile, u32 (&x)[32], int tau)
{
    constexpr int T = Cfg32<LOGN>::T;
#pragma unroll
    for (int m = 0; m < 32; m++) x[m] = (u32)tile[tau + pos32(T * m)];
}

// FQ_KEYBM: key product against a residue table prepared per launch (base multiplication, policies with AR::BASEMUL)
enum { FQ_POLYMUL = 0, FQ_KEY16 = 1, FQ_KEY32 = 2, FQ_KEYBM = 3 };

// reference NTT-domain index of the thread's pass-1 element e (position 32 tau + e of the bit-reversed order):
// brev(32 tau + e) = brev5(e) << (LOGN - 5) | brev_{LOGN-5}(tau); for fixed e the lanes of a polynomial read
// n/32 consecutive coefficients
template <int LOGN>
__device__ __forceinline__ int ntt_index(int tau, int e)
{
    return (int)((__brev((unsigned)e) >> 27) << (LOGN - 5)) | (int)(__brev((unsigned)tau) >> (32 - (LOGN - 5)));
}


template <class AR>
struct W32Const {
    const int32_t *pf;                           // pass-1 forward table, thread-major (slot32): WORDS arrays of n words
    const int32_t *pi;                           // pass-1 inverse table
    const int32_t *pz;                           // base multiplication: (w, wq) of zeta for the thread's 8 blocks of four,
                                                 // [pair of blocks][tau][4 words] (policies with AR::BASEMUL)
    typename AR::E f0[31], i0[31];               // entries 1..31: stages 0..4
    typename AR::E ninv, one;
    typename AR::K k;
    int32_t q, nq, x0;
    uint32_t M;                                  // floor(2^32 / q): 32-bit Barrett of the out-of-range path
    int r0;                                      // bit 0: reduce every coefficient at the entry of inverse pass 0;
                                                 // bit 1: reduce the second operand before the pointwise product
};

template <class AR>
struct W32 {
using Const = W32Const<AR>;
using E = typename AR::E;


static __device__ __forceinline__ int32_t bred(int32_t p, const Const &c)
{
    const int32_t qe = (int32_t)(((int64_t)p * (int64_t)c.M + 0x80000000ll) >> 32);
    return qe * c.nq + p;
}
static __device__ __forceinline__ bool out_of_range(int32_t v, const Const &c)
{
    return ((u32)v + (u32)c.x0) > (u32)(2 * c.x0);
}

// ---- pass 0: stages 0..4 on x[m] = element tau + T m ---------------------------------------------------
static __device__ __forceinline__ void fwd_pass0(u32 (&x)[32], const Const &c)
{
    if constexpr (AR::PASS0_IMM) { AR::fwd_pass0(x, c.k); return; }
#pragma unroll
    for (int s = 0; s < 5; s++) {
        const int half = 16 >> s;
#pragma unroll
        for (int m = 0; m < 32; m++)
            if ((m & half) == 0) {
                if (s == 0) AR::ct0(x[m], x[m + half], AR::cb(c.f0[0]), c.k);      // x[0..15] arrive raw (load_operand)
                else        AR::ct(x[m], x[m + half], AR::cb(c.f0[(1 << s) - 1 + (m >> (5 - s))]), c.k);
            }
    }
}

// stages 4..1, then stage 0 with n^-1 folded into both branches; returns canonical residues
static __device__ __forceinline__ void inv_pass0(u32 (&x)[32], const Const &c)
{
    if constexpr (AR::PASS0_IMM) { AR::inv_pass0(x, c.k); return; }
#pragma unroll
    for (int s = 4; s >= 1; s--) {
        const int half = 16 >> s;
#pragma unroll
        for (int m = 0; m < 32; m++)
            if ((m & half) == 0) AR::gs(x[m], x[m + half], AR::cb(c.i0[(1 << s) - 1 + (m >> (5 - s))]), c.k);
    }
#pragma unroll
    for (int m = 0; m < 16; m++) AR::fin(x[m], x[m + 16], c.ninv, c.i0[0], c.k);
}

// ---- pass 1 -------------------------------------------------------------------------------------------
// CNT consecutive entries r0 .. r0 + CNT - 1 of thread tau for stage S (CNT in 1, 2, 4)
template <int LOGN, int S, int CNT>
static __device__ __forceinline__ void load_entries(E (&tw)[CNT], const int32_t *tab, int tau, int r0)
{
    using C = Cfg32<LOGN>;
    constexpr int LEN = C::N >> (S + 1);
    constexpr int G = 16 / LEN;
    constexpr int V = G < 4 ? G : 4;
    constexpr int N = C::N;
    constexpr int W = AR::WORDS;                    // parallel arrays of n words each
    const int32_t *p = tab + (1 << S) + ((r0 / V) * C::T + tau) * V + (r0 % V);
    if constexpr (CNT == 4) {
        int4 v[W];
#pragma unroll
        for (int k = 0; k < W; k++) v[k] = __ldg(reinterpret_cast<const int4 *>(p + k * N));
        int32_t wx[4], wy[4], wz[4], ww[4];
#pragma unroll
        for (int k = 0; k < W; k++) { wx[k] = v[k].x; wy[k] = v[k].y; wz[k] = v[k].z; ww[k] = v[k].w; }
        tw[0] = AR::mk(wx); tw[1] = AR::mk(wy); tw[2] = AR::mk(wz); tw[3] = AR::mk(ww);
    } else if constexpr (CNT == 2) {
        int2 v[W];
#pragma unroll
        for (int k = 0; k < W; k++) v[k] = __ldg(reinterpret_cast<const int2 *>(p + k * N));
        int32_t wx[4], wy[4];
#pragma unroll
        for (int k = 0; k < W; k++) { wx[k] = v[k].x; wy[k] = v[k].y; }
        tw[0] = AR::mk(wx); tw[1] = AR::mk(wy);
    } else {
        int32_t wx[4];
#pragma unroll
        for (int k = 0; k < W; k++) wx[k] = __ldg(p + k * N);
        tw[0] = AR::mk(wx);
    }
}

// one radix-2 stage S (forward: Cooley-Tukey, inverse: Gentleman-Sande) on sub-chunk h of NOPS operands
// UNB (forward only): the butterflies emit unbiased values (the stage in front of the base multiplication)
template <int LOGN, int S, int NOPS, bool INV, int CH, bool UNB = false>
static __device__ __forceinline__ void stage1(u32 (&xa)[CH], u32 (&xb)[CH], const Const &c, int tau, int h)
{
    using C = Cfg32<LOGN>;
    constexpr int LEN = C::N >> (S + 1);
    constexpr int CNT = CH / (2 * LEN);              // twiddles of this (sub-)chunk in this stage
    constexpr int GRP = CNT < 4 ? CNT : 4;
    const int32_t *tab = INV ? c.pi : c.pf;
#pragma unroll
    for (int g0 = 0; g0 < CNT; g0 += GRP) {
        E tw[GRP];
        load_entries<LOGN, S, GRP>(tw, tab, tau, h * CNT + g0);
#pragma unroll
        for (int g = 0; g < GRP; g++) {
#pragma unroll
            for (int j = 0; j < LEN; j++) {
                const int i = (g0 + g) * 2 * LEN + j;
                if (INV) {
                    AR::gs(xa[i], xa[i + LEN], tw[g], c.k);
                } else if constexpr (UNB) {
                    AR::ct_unb(xa[i], xa[i + LEN], tw[g], c.k);
                    if (NOPS == 2) AR::ct_unb(xb[i], xb[i + LEN], tw[g], c.k);
                } else {
                    AR::ct(xa[i], xa[i + LEN], tw[g], c.k);
                    if (NOPS == 2) AR::ct(xb[i], xb[i + LEN], tw[g], c.k);
                }
            }
        }
    }
}

template <int LOGN, int S, int NOPS>
static __device__ __forceinline__ void fwd_stages1(u32 (&xa)[Cfg32<LOGN>::SUB], u32 (&xb)[Cfg32<LOGN>::SUB],
                                            const Const &c, int tau, int h)
{
    if constexpr (S < LOGN) {
        stage1<LOGN, S, NOPS, false, Cfg32<LOGN>::SUB>(xa, xb, c, tau, h);
        fwd_stages1<LOGN, S + 1, NOPS>(xa, xb, c, tau, h);
    }
}
// forward stages S .. LOGN - 3 of NOPS operands, the last one emitting unbiased values
template <int LOGN, int S, int NOPS = 2>
static __device__ __forceinline__ void fwd_stages1_bm(u32 (&xa)[Cfg32<LOGN>::SUB], u32 (&xb)[Cfg32<LOGN>::SUB],
                                               const Const &c, int tau, int h)
{
    if constexpr (S < LOGN - 3) {
        stage1<LOGN, S, NOPS, false, Cfg32<LOGN>::SUB>(xa, xb, c, tau, h);
        fwd_stages1_bm<LOGN, S + 1, NOPS>(xa, xb, c, tau, h);
    } else {
        stage1<LOGN, S, NOPS, false, Cfg32<LOGN>::SUB, true>(xa, xb, c, tau, h);
    }
}
// xa <- xa * key modulo X^4 - zeta for the SUB / 4 blocks of sub-chunk h; kres = the launch's residue table,
// 16 words per block as four 128-bit vectors [b | float b | zeta b | float zeta b]; vector v of block j of thread tau
// at ((4 j + v) T + tau) 4: the lanes of a polynomial read contiguous 16-byte words
template <int LOGN>
static __device__ __forceinline__ void keymul_sub(u32 (&xa)[Cfg32<LOGN>::SUB], const int32_t *kres, const Const &c, int tau, int h)
{
    using C = Cfg32<LOGN>;
    constexpr int GROUPS = C::SUB / 4;
#pragma unroll
    for (int g = 0; g < GROUPS; g++) {
        const int4 *p = reinterpret_cast<const int4 *>(kres) + (h * GROUPS + g) * 4 * C::T + tau;
        AR::bmk4(&xa[4 * g], __ldg(p), __ldg(p + C::T), __ldg(p + 2 * C::T), __ldg(p + 3 * C::T), c.k);
    }
}
// xa <- xa * xb modulo X^4 - zeta for the SUB / 4 blocks of sub-chunk h (fq_arith.cuh: basemul4)
template <int LOGN>
static __device__ __forceinline__ void basemul_sub(u32 (&xa)[Cfg32<LOGN>::SUB], const u32 (&xb)[Cfg32<LOGN>::SUB],
                                            const Const &c, int tau, int h)
{
    using C = Cfg32<LOGN>;
    constexpr int PAIRS = C::SUB / 8;
#pragma unroll
    for (int pr = 0; pr < PAIRS; pr++) {
        const int4 z = __ldg(reinterpret_cast<const int4 *>(c.pz) + (h * PAIRS + pr) * C::T + tau);
        AR::bm4(&xa[8 * pr], &xb[8 * pr], z.x, z.y, c.k);
        AR::bm4(&xa[8 * pr + 4], &xb[8 * pr + 4], z.z, z.w, c.k);
    }
}

template <int LOGN, int S>
static __device__ __forceinline__ void inv_stages1(u32 (&x)[Cfg32<LOGN>::SUB], const Const &c, int tau, int h)
{
    if constexpr (S >= Cfg32<LOGN>::S1) {
        stage1<LOGN, S, 1, true, Cfg32<LOGN>::SUB>(x, x, c, tau, h);
        inv_stages1<LOGN, S - 1>(x, c, tau, h);
    }
}

// n = 1024 only: stage 5 (forward) / its inverse on the thread's whole 32-element chunk, in place in the tile
template <int LOGN, bool INV>
static __device__ __forceinline__ void chunk_stage5(int32_t *p, const Const &c, int tau)
{
    if constexpr (Cfg32<LOGN>::S1 > 5) {
        u32 x[32];
        load_sub<32>(p, x);
        stage1<LOGN, 5, 1, INV, 32>(x, x, c, tau, 0);
        store_sub<32>(p, x);
    }
}

// CHK = false: the caller vouches for |coefficient| <= c.x0 (SCGPU_PLAN_INPUTS_IN_RANGE); no range vote
template <int LOGN, bool CHK = true>
static __device__ __forceinline__ void load_operand(u32 (&x)[32], const int32_t *row, int tau, const Const &c)
{
    constexpr int T = Cfg32<LOGN>::T;
    int32_t v[32];
    bool wide = false;
#pragma unroll
    for (int m = 0; m < 32; m++) {
        v[m] = __ldg(row + tau + m * T);
        if (CHK) wide |= out_of_range(v[m], c);
    }
    if (CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
        for (int m = 0; m < 32; m++) v[m] = bred(v[m], c);
    }
    // the low half stays raw: stage 0 of fwd_pass0 (AR::ct0) encodes it inside its own adds
#pragma unroll
    for (int m = 0; m < 32; m++) x[m] = m < 16 ? (u32)v[m] : AR::enc(v[m]);
}

// same, from a raw row that a bulk copy (TMA) has staged at the start of the tile region
template <int LOGN, bool CHK = true>
static __device__ __forceinline__ void load_operand_staged(u32 (&x)[32], const int32_t *raw, int tau, const Const &c)
{
    constexpr int T = Cfg32<LOGN>::T;
    int32_t v[32];
    bool wide = false;
#pragma unroll
    for (int m = 0; m < 32; m++) {
        v[m] = raw[tau + m * T];
        if (CHK) wide |= out_of_range(v[m], c);
    }
    if (CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
        for (int m = 0; m < 32; m++) v[m] = bred(v[m], c);
    }
    // the low half stays raw: stage 0 of fwd_pass0 (AR::ct0) encodes it inside its own adds
#pragma unroll
    for (int m = 0; m < 32; m++) x[m] = m < 16 ? (u32)v[m] : AR::enc(v[m]);
}

// ---- the addend of the *_add entry points:  out = (product + e) mod q ----------------------------------------------
// x in [0, q), |v| <= 4 q:  t = x + v + 4 q lies in [0, 9 q) (< 2^31 for q < 2^27); with M = floor(2^32 / q) the
// quotient floor(t M / 2^32) is floor(t / q) or one less (t (2^32 / q - M) < 2^32), so t minus it times q lies in
// [0, 2 q) and one conditional -q is canonical.  IADD3, IMAD.HI, IMAD, IADD, VIMNMX per coefficient.
static __device__ __forceinline__ u32 add_canon(u32 x, int32_t v, u32 q4, const Const &c)
{
    const u32 t = x + (u32)v + q4;
    const u32 r = __umulhi(t, c.M) * (u32)c.nq + t;
    return min(r, r - (u32)c.q);
}
// x[m] = canonical residue of element tau + T m of a row  ->  (x[m] + erow[tau + T m]) mod q.  The lane reads the
// addresses it stores to (for each m the T lanes of a polynomial read T consecutive words: whole sectors, any
// alignment).  CHK: a warp vote on |e| > 4 q, then the Barrett reduction of the out-of-range path (|bred(e)| <= q);
// without it the caller vouches |e| <= 4 q.  (32 addend words next to the 32 results spill nothing, k_matvec16_w32
// included: its accumulators are dead once the inverse transform has run.)
template <int LOGN, bool CHK>
static __device__ __forceinline__ void add_addend(u32 (&x)[32], const int32_t *erow, int tau, const Const &c)
{
    constexpr int T = Cfg32<LOGN>::T;
    const u32 q4 = 4u * (u32)c.q;
    int32_t v[32];
    bool wide = false;
#pragma unroll
    for (int m = 0; m < 32; m++) {
        v[m] = erow[tau + m * T];
        if (CHK) wide |= (u32)v[m] + q4 > 2u * q4;
    }
    if (CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
        for (int m = 0; m < 32; m++) v[m] = bred(v[m], c);
    }
#pragma unroll
    for (int m = 0; m < 32; m++) x[m] = add_canon(x[m], v[m], q4, c);
}

};  // struct W32

// The addend rows of an iteration are requested into L2 when it starts (one 128-byte line per lane: the n/32 lanes of a
// row cover its 4 n bytes), so that the loads of the epilogue find them there.  Every address lies inside an addend
// row (rows beyond the batch are clamped to row 0, as the operands are).
__device__ __forceinline__ void prefetch_l2(const int32_t *p)
{
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// TMA = true: operand rows arrive by bulk copy (16-byte aligned rows); false: plain LDG (any alignment)
// BM = true (FQ_POLYMUL, policies with AR::BASEMUL): the transforms stop two stages early and the residues modulo
// X^4 - zeta are multiplied directly (c carries the last-stage entries for (n/4)^-1).  CHK = false: no range vote.
// ADD: out = (product + e) mod q, e [count][n] (may be out itself); without it e is not read.
template <class AR, int LOGN, int MODE, bool TMA, bool BM = false, bool CHK = true, bool ADD = false>
__global__ void __launch_bounds__(kThreads32, FQ32_MINB)
k_polymul_w32(int32_t *__restrict__ out, const int32_t *__restrict__ a, const void *__restrict__ bsrc,
               size_t b_stride, size_t count, unsigned long long *ctr, const __grid_constant__ W32Const<AR> c,
               const int32_t *e)
{
    using C = Cfg32<LOGN>;
    using W = W32<AR>;
    constexpr int N = C::N, T = C::T, SUB = C::SUB;
    __shared__ __align__(16) int32_t tiles[2][C::POLYS][C::TS];      // slot stride TS = T (mod 32) banks
    const int lane = threadIdx.x & 31;
    const int tau = lane % T;
    const int slot = (threadIdx.x / 32) * C::PW + lane / T;       // polynomial slot inside the CTA
    int32_t *ta = tiles[0][slot];
    int32_t *tb = tiles[1][slot];
    // bulk-copy pipeline state: bars[warp][0 / 1] complete when the a / b rows of the warp's next product have
    // landed; `other` = byte offset between a polynomial's two tile regions, whose roles swap every iteration
    __shared__ __align__(8) uint64_t bars[kThreads32 / 32][2];
    const int warp = threadIdx.x / 32;
    uint32_t parity = 0;
    constexpr uint32_t ROW_BYTES = (uint32_t)N * 4u;
    auto fetch = [&](int op, size_t nbase, int32_t *region0) {
        // lane 0: rows of the warp's PW polynomials of the product group starting at nbase -> region0[p]
        mbar_expect_tx(&bars[warp][op], ROW_BYTES * C::PW);
#pragma unroll
        for (int p = 0; p < C::PW; p++) {
            size_t row = nbase + (size_t)warp * C::PW + p;
            if (row >= count) row = 0;
            const int32_t *src = op == 0 ? a + row * N : static_cast<const int32_t *>(bsrc) + row * b_stride;
            bulk_g2s(region0 + p * C::TS, src, ROW_BYTES, &bars[warp][op]);
        }
    };
    const size_t first = (size_t)blockIdx.x * C::POLYS;
    if (TMA) {
        if (lane == 0) {
            mbar_init(&bars[warp][0], 1);
            mbar_init(&bars[warp][1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if (lane == 0 && first < count) {
            fetch(0, first, tiles[0][warp * C::PW]);
            if (MODE == FQ_POLYMUL) fetch(1, first, tiles[1][warp * C::PW]);
        }
    }

    Claim cl;
    for (cl.init(ctr, (unsigned)((count + C::POLYS - 1) / C::POLYS)); (size_t)cl.g * C::POLYS < count;) {
        const size_t base = (size_t)cl.g * C::POLYS;
        const size_t poly = base + slot;
        const bool live = poly < count;
        const size_t prow = live ? poly : 0;
        cl.issue(ctr, lane);
        const size_t nbase = (size_t)cl.gn * C::POLYS;
        if (ADD) prefetch_l2(e + prow * N + 32 * tau);
        // rolled loops (operand, sub-chunk): the fully unrolled body was 60 KB of SASS and spent 2 of every
        // 7 stall cycles waiting for instructions (profiles/polymul_r02c_*); the L1.5 I-cache holds 32 KB
#pragma unroll 1
        for (int op = 0; op < (MODE == FQ_POLYMUL ? 2 : 1); op++) {
            u32 x[32];
            int32_t *tile = op == 0 ? ta : tb;
            if (TMA) {
                mbar_wait(&bars[warp][op], parity);
                if (MODE != FQ_POLYMUL) {
                    // key product: only one operand streams, so the other region is free for the WHOLE iteration --
                    // the next product's rows are put in flight a full iteration ahead (its group is known: Claim)
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0 && nbase < count) fetch(0, nbase, tb - (lane / T) * C::TS);
                }
                W::template load_operand_staged<LOGN, CHK>(x, tile, tau, c);
                __syncwarp();                     // the padded result overwrites the raw row in place
            } else {
                const int32_t *row = op == 0 ? a + prow * N : static_cast<const int32_t *>(bsrc) + prow * b_stride;
                W::template load_operand<LOGN, CHK>(x, row, tau, c);
            }
            W::fwd_pass0(x, c);
            store_pass0<LOGN>(tile, x, tau);
        }
        __syncwarp();
        if constexpr (C::S1 > 5) {
#pragma unroll 1
            for (int op = 0; op < (MODE == FQ_POLYMUL ? 2 : 1); op++) W::template chunk_stage5<LOGN, false>((op == 0 ? ta : tb) + 36 * tau, c, tau);
        }
#pragma unroll 1
        for (int h = 0; h < C::NSUB; h++) {
            u32 xa[SUB], xb[SUB];
            int32_t *pa = ta + 36 * tau + SUB * h;
            load_sub<SUB>(pa, xa);
            if constexpr (MODE == FQ_KEYBM) {
                static_assert(MODE != FQ_KEYBM || BM, "the residue-table key product is a base multiplication");
                W::template fwd_stages1_bm<LOGN, C::S1, 1>(xa, xb, c, tau, h);
                W::template keymul_sub<LOGN>(xa, static_cast<const int32_t *>(bsrc), c, tau, h);
            } else if constexpr (MODE == FQ_POLYMUL && BM) {
                load_sub<SUB>(tb + 36 * tau + SUB * h, xb);
                W::template fwd_stages1_bm<LOGN, C::S1>(xa, xb, c, tau, h);
                W::template basemul_sub<LOGN>(xa, xb, c, tau, h);
            } else if constexpr (MODE == FQ_POLYMUL) {
                load_sub<SUB>(tb + 36 * tau + SUB * h, xb);
                W::template fwd_stages1<LOGN, C::S1, 2>(xa, xb, c, tau, h);
                if (c.r0 & 2) {                                      // 26-bit moduli: lazy x lazy leaves the Montgomery range
#pragma unroll
                    for (int i = 0; i < SUB; i++) xb[i] = AR::red(xb[i], c.one, c.k);
                }
#pragma unroll
                for (int i = 0; i < SUB; i++)
                    xa[i] = AR::pw(xa[i], xb[i], c.k);
            } else {
                W::template fwd_stages1<LOGN, C::S1, 1>(xa, xb, c, tau, h);
                int32_t kv[SUB];
                bool wide = false;
                // ntt_index(tau, SUB h + i) = (brev5(i) + brev5(SUB h)) << (LOGN - 5) | brev(tau): the low bits
                // of the 5-bit field come from i (compile time), the high ones from h -- one base per sub-chunk,
                // immediate offsets per element
                const size_t kbase = prow * b_stride + (size_t)ntt_index<LOGN>(tau, SUB * h);
#pragma unroll
                for (int i = 0; i < SUB; i++) {
                    const int off = (int)((__brev((unsigned)i) >> 27) << (LOGN - 5));
                    if (MODE == FQ_KEY16) kv[i] = (int32_t)__ldg(static_cast<const int16_t *>(bsrc) + kbase + off);
                    else {
                        kv[i] = __ldg(static_cast<const int32_t *>(bsrc) + kbase + off);
                        if (CHK) wide |= W::out_of_range(kv[i], c);
                    }
                }
                if (CHK && MODE == FQ_KEY32 && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                    for (int i = 0; i < SUB; i++) kv[i] = W::bred(kv[i], c);
                }
#pragma unroll
                for (int i = 0; i < SUB; i++)
                    xa[i] = AR::pwraw(xa[i], kv[i], c.k);
            }
            W::template inv_stages1<LOGN, BM ? LOGN - 3 : LOGN - 1>(xa, c, tau, h);
            store_sub<SUB>(pa, xa);
        }
        W::template chunk_stage5<LOGN, true>(ta + 36 * tau, c, tau);
        if (TMA) fence_proxy_async();
        __syncwarp();
        // tb is free from here on: the next product's a rows go there
        if (TMA && MODE == FQ_POLYMUL && lane == 0 && nbase < count) fetch(0, nbase, tb - (lane / T) * C::TS);
        {
            u32 x[32];
            load_pass0<LOGN>(ta, x, tau);
            if (TMA && MODE == FQ_POLYMUL) {
                fence_proxy_async();
                __syncwarp();
                // every coefficient is in registers: ta takes the next product's b rows
                if (lane == 0 && nbase < count) fetch(1, nbase, ta - (lane / T) * C::TS);
            }
            if (c.r0 & 1) {
#pragma unroll
                for (int m = 0; m < 32; m++) x[m] = AR::red(x[m], c.one, c.k);
            }
            W::inv_pass0(x, c);
            if (ADD) W::template add_addend<LOGN, CHK>(x, e + prow * N, tau, c);
            if (live) {
                int32_t *orow = out + poly * N;
#pragma unroll
                for (int m = 0; m < 32; m++) orow[tau + m * T] = (int32_t)x[m];
            }
        }
        if (TMA) {
            int32_t *t = ta; ta = tb; tb = t;         // the regions swap roles
            parity ^= 1u;
        } else {
            __syncwarp();
        }
        cl.advance(ctr);
    }
}


// ---- single transforms with CANONICAL output ---------------------------------------------------------------------
//   INV = false:  out = normalize_32(fwd_ntt_32_16/32(a))   residues in [0, q), the reference's NTT-domain order
//   INV = true :  out = inv_ntt_32_16/32(a)                 a in the reference's NTT-domain order, any SINT32
// Both results are canonical in the reference, so the arithmetic inside is free (as for the fused products); the
// variant-exact kernels of ntt_exact.cu remain the way to get fwd_ntt's lazily reduced representative itself.
// TMA = true: the next polynomial's row is bulk-copied into a staging row while the current one is transformed
// (16-byte aligned rows); false: plain loads.
template <class AR, int LOGN, bool INV, bool TMA, bool CHK = true>
__global__ void __launch_bounds__(kThreads32, FQ32_MINB)
k_ntt_w32(int32_t *__restrict__ out, const int32_t *__restrict__ a, size_t count, unsigned long long *ctr,
          const __grid_constant__ W32Const<AR> c)
{
    using C = Cfg32<LOGN>;
    using W = W32<AR>;
    constexpr int N = C::N, T = C::T, SUB = C::SUB;
    constexpr int AROW = N + T;                                      // staging row stride: T banks between polynomials
    constexpr uint32_t ROW_BYTES = (uint32_t)N * 4u;
    __shared__ __align__(16) int32_t tiles[C::POLYS][C::TS];
    __shared__ __align__(16) int32_t stage_rows[TMA ? C::POLYS : 1][AROW];
    __shared__ __align__(8) uint64_t bars[kThreads32 / 32];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x / 32;
    const int tau = lane % T;
    const int slot = warp * C::PW + lane / T;
    int32_t *tile = tiles[slot];
    const int32_t *stage = stage_rows[TMA ? slot : 0];
    const int taurev = (int)(__brev((unsigned)tau) >> (32 - (LOGN - 5)));
    uint32_t parity = 0;
    auto fetch = [&](size_t nbase) {                                 // lane 0: rows of the warp's PW polynomials
        mbar_expect_tx(&bars[warp], ROW_BYTES * C::PW);
        for (int p = 0; p < C::PW; p++) {
            size_t row = nbase + (size_t)warp * C::PW + p;
            if (row >= count) row = 0;
            bulk_g2s(stage_rows[TMA ? warp * C::PW + p : 0], a + row * N, ROW_BYTES, &bars[warp]);
        }
    };
    const size_t first = (size_t)blockIdx.x * C::POLYS;
    if (TMA) {
        if (lane == 0) {
            mbar_init(&bars[warp], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if (lane == 0 && first < count) fetch(first);
    }

    Claim cl;
    for (cl.init(ctr, (unsigned)((count + C::POLYS - 1) / C::POLYS)); (size_t)cl.g * C::POLYS < count;) {
        const size_t base = (size_t)cl.g * C::POLYS;
        const size_t poly = base + slot;
        const bool live = poly < count;
        const size_t prow = live ? poly : 0;
        cl.issue(ctr, lane);
        const size_t nbase = (size_t)cl.gn * C::POLYS;
        if (!INV) {
            {
                u32 x[32];
                if (TMA) {
                    mbar_wait(&bars[warp], parity); parity ^= 1u;
                    W::template load_operand_staged<LOGN, CHK>(x, stage, tau, c);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0 && nbase < count) fetch(nbase);    // the staging row is in registers
                } else {
                    W::template load_operand<LOGN, CHK>(x, a + prow * N, tau, c);
                }
                W::fwd_pass0(x, c);
                store_pass0<LOGN>(tile, x, tau);
            }
            __syncwarp();
            W::template chunk_stage5<LOGN, false>(tile + 36 * tau, c, tau);
#pragma unroll 1
            for (int h = 0; h < C::NSUB; h++) {
                u32 xa[SUB], xb[SUB];
                load_sub<SUB>(tile + 36 * tau + SUB * h, xa);
                W::template fwd_stages1<LOGN, C::S1, 1>(xa, xb, c, tau, h);
                int32_t *orow = out + poly * N + ntt_index<LOGN>(tau, SUB * h);
#pragma unroll
                for (int i = 0; i < SUB; i++) {
                    u32 v = (u32)AR::dec(AR::red(xa[i], c.one, c.k));           // in (-q, q + q/16)
                    v = min(v, v + (u32)c.q);
                    v = min(v, v - (u32)c.q);
                    if (live) orow[(int)((__brev((unsigned)i) >> 27) << (LOGN - 5))] = (int32_t)v;
                }
            }
            __syncwarp();
        } else {
            if (TMA) { mbar_wait(&bars[warp], parity); parity ^= 1u; }
#pragma unroll 1
            for (int h = 0; h < C::NSUB; h++) {
                int32_t v[SUB];
                bool wide = false;
                if (TMA) {
                    const int32_t *irow = stage + ntt_index<LOGN>(tau, SUB * h);
#pragma unroll
                    for (int i = 0; i < SUB; i++) {
                        v[i] = irow[(int)((__brev((unsigned)i) >> 27) << (LOGN - 5))];
                        if (CHK) wide |= W::out_of_range(v[i], c);
                    }
                } else {
                    const int32_t *irow = a + prow * N + ntt_index<LOGN>(tau, SUB * h);
#pragma unroll
                    for (int i = 0; i < SUB; i++) {
                        v[i] = __ldg(irow + (int)((__brev((unsigned)i) >> 27) << (LOGN - 5)));
                        if (CHK) wide |= W::out_of_range(v[i], c);
                    }
                }
                if (CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                    for (int i = 0; i < SUB; i++) v[i] = W::bred(v[i], c);
                }
                u32 x[SUB];
#pragma unroll
                for (int i = 0; i < SUB; i++) x[i] = AR::red(AR::enc(v[i]), c.one, c.k);   // the bounds assume reduced input
                W::template inv_stages1<LOGN, LOGN - 1>(x, c, tau, h);
                store_sub<SUB>(tile + 36 * tau + SUB * h, x);
            }
            if (TMA) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0 && nbase < count) fetch(nbase);        // every sub-chunk has been read
            }
            W::template chunk_stage5<LOGN, true>(tile + 36 * tau, c, tau);
            __syncwarp();
            {
                u32 x[32];
                load_pass0<LOGN>(tile, x, tau);
                if (c.r0 & 1) {
#pragma unroll
                    for (int m = 0; m < 32; m++) x[m] = AR::red(x[m], c.one, c.k);
                }
                W::inv_pass0(x, c);
                if (live) {
                    int32_t *orow = out + poly * N;
#pragma unroll
                    for (int m = 0; m < 32; m++) orow[tau + m * T] = (int32_t)x[m];
                }
            }
            __syncwarp();
        }
        cl.advance(ctr);
    }
    (void)taurev;
}

// ---- module-LWE matrix-vector product  t_i = INTT(sum_j A_ij o NTT(s_j))  (module_lwe.c:588-748) -------------
// Same warp-local schedule.  The l transformed vectors stay in shared memory (padded pass-1 layout, unbiased),
// each output row accumulates its l pointwise products in registers.  HBM traffic is dominated by A
// (k l rows per instance against l + k for s and t), so with TMA = true every row moves by bulk copy:
//   * A_ij rows (contiguous n words) land in a one-row staging buffer per instance; as soon as a thread group
//     has pulled its 32 coefficients into registers the next row (or the next instance's first row) is in
//     flight, i.e. a row's DRAM latency is covered by one whole pointwise step;
//   * the next instance's s rows are fetched into the stash tiles during the last inverse transform.
// The reference's NTT-domain order is our bit-reversed one: element e of thread tau is coefficient
// brev5(e) * (n/32) + brev(tau) of the row (ntt_index), so for a fixed e the lanes of an instance read n/32
// consecutive words: conflict-free from the staging row (instances 8 banks apart), one full sector from HBM
// in the LDG variant.
// SHARED_A: one matrix [k][l][n] for every instance (scgpu_matvec_shared_batch), addressed with an instance stride of 0
// ADD: t_i = (t_i + e_i) mod q, e [count][k][n] (may be out itself); without it e is not read.
template <class AR, int LOGN, bool TMA, bool CHK = true, bool SHARED_A = false, bool ADD = false>
__global__ void __launch_bounds__(kThreads32)
k_matvec_w32(int32_t *__restrict__ out, const int32_t *__restrict__ A, const int32_t *__restrict__ s,
              int k, int l, size_t count, unsigned long long *ctr, const __grid_constant__ W32Const<AR> c,
              const int32_t *e)
{
    using C = Cfg32<LOGN>;
    using W = W32<AR>;
    constexpr int N = C::N, T = C::T, SUB = C::SUB, NSUB = C::NSUB;
    constexpr int AROW = N + T;                                      // staging row stride: T banks between instances
    constexpr uint32_t ROW_BYTES = (uint32_t)N * 4u;
    extern __shared__ __align__(16) int32_t dyn_tiles[];             // [l + 1][POLYS][TS], then [POLYS][AROW]
    __shared__ __align__(8) uint64_t bars[kThreads32 / 32][3];       // [warp][0: s rows, 1: A rows in S, 2: A rows in X]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x / 32;
    const int tau = lane % T;
    const int slot = warp * C::PW + lane / T;
    int32_t *xt = dyn_tiles + slot * C::TS;                          // exchange tile of the inverse transform
    int32_t *astage = dyn_tiles + (size_t)(l + 1) * C::POLYS * C::TS + slot * AROW;
    const int taurev = (int)(__brev((unsigned)tau) >> (32 - (LOGN - 5)));
    // Two A rows in flight without more shared memory: even columns j of the matrix travel through the staging rows S,
    // odd columns through X = the exchange tile of the inverse transform, which is idle while a row accumulates.  X takes
    // its next row only after the inverse transform of the output row has finished (S carries the row in flight across
    // it).  One row in flight left a warp waiting for DRAM in 21 % of its stall samples at 8 warps per SM
    // (profiles/dil_matvec_r2_ncu.json); a second staging buffer proper costs a CTA per SM and was slower.
    const int32_t *xstage = dyn_tiles + slot * AROW;
    uint32_t par_s = 0, par_a0 = 0, par_a1 = 0;

    // lane 0: rows of the warp's PW instances (clamped to instance 0 beyond the batch)
    auto fetch_s = [&](size_t nbase) {
        mbar_expect_tx(&bars[warp][0], ROW_BYTES * C::PW * (uint32_t)l);
        for (int p = 0; p < C::PW; p++) {
            size_t row = nbase + (size_t)warp * C::PW + p;
            if (row >= count) row = 0;
            for (int j = 0; j < l; j++)
                bulk_g2s(dyn_tiles + ((size_t)(j + 1) * C::POLYS + warp * C::PW + p) * C::TS, s + (row * l + j) * N, ROW_BYTES, &bars[warp][0]);
        }
    };
    auto fetch_a = [&](size_t nbase, int step, int which) {
        mbar_expect_tx(&bars[warp][1 + which], ROW_BYTES * C::PW);
        int32_t *dst = which ? dyn_tiles : dyn_tiles + (size_t)(l + 1) * C::POLYS * C::TS;
        for (int p = 0; p < C::PW; p++) {
            size_t row = nbase + (size_t)warp * C::PW + p;
            if (row >= count) row = 0;
            bulk_g2s(dst + (warp * C::PW + p) * AROW, A + ((SHARED_A ? (size_t)0 : row * k * l) + step) * N, ROW_BYTES, &bars[warp][1 + which]);
        }
    };
    const size_t first = (size_t)blockIdx.x * C::POLYS;
    if (TMA) {
        if (lane == 0) {
            mbar_init(&bars[warp][0], 1);
            mbar_init(&bars[warp][1], 1);
            mbar_init(&bars[warp][2], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if (lane == 0 && first < count) { fetch_s(first); fetch_a(first, 0, 0); if (l >= 2) fetch_a(first, 1, 1); }
    }

    Claim cl;
    for (cl.init(ctr, (unsigned)((count + C::POLYS - 1) / C::POLYS)); (size_t)cl.g * C::POLYS < count;) {
        const size_t base = (size_t)cl.g * C::POLYS;
        const size_t inst = base + slot;
        const bool live = inst < count;
        const size_t irow = live ? inst : 0;
        cl.issue(ctr, lane);
        const size_t nbase = (size_t)cl.gn * C::POLYS;
        if (ADD) {
            for (int i = 0; i < k; i++) prefetch_l2(e + (irow * k + i) * N + 32 * tau);
        }
        if (TMA) { mbar_wait(&bars[warp][0], par_s); par_s ^= 1u; }
#pragma unroll 1
        for (int j = 0; j < l; j++) {
            u32 x[32];
            int32_t *tile = dyn_tiles + ((size_t)(j + 1) * C::POLYS + slot) * C::TS;
            if (TMA) {
                W::template load_operand_staged<LOGN, CHK>(x, tile, tau, c);
                __syncwarp();
            } else {
                W::template load_operand<LOGN, CHK>(x, s + (irow * l + j) * N, tau, c);
            }
            W::fwd_pass0(x, c);
            store_pass0<LOGN>(tile, x, tau);
        }
        __syncwarp();
#pragma unroll 1
        for (int j = 0; j < l; j++) {
#pragma unroll 1
            for (int h = 0; h < NSUB; h++) {
                u32 xa[SUB], xb[SUB];
                int32_t *p = dyn_tiles + ((size_t)(j + 1) * C::POLYS + slot) * C::TS + 36 * tau + SUB * h;
                load_sub<SUB>(p, xa);
                W::template fwd_stages1<LOGN, C::S1, 1>(xa, xb, c, tau, h);
#pragma unroll
                for (int i = 0; i < SUB; i++) xa[i] = (u32)AR::dec(xa[i]);
                store_sub<SUB>(p, xa);                               // only this thread reads it again
            }
        }
#pragma unroll 1
        for (int i = 0; i < k; i++) {
            typename AR::Acc part[32];
#pragma unroll
            for (int e = 0; e < 32; e++) part[e] = AR::acc_zero();
#pragma unroll 1
            for (int j = 0; j < l; j++) {
                int32_t av[32];
                bool wide = false;
                if (TMA) {
                    const int which = j & 1;
                    if (which) { mbar_wait(&bars[warp][2], par_a1); par_a1 ^= 1u; }
                    else       { mbar_wait(&bars[warp][1], par_a0); par_a0 ^= 1u; }
                    const int32_t *arow = which ? xstage : astage;
#pragma unroll
                    for (int e = 0; e < 32; e++) {
                        av[e] = arow[taurev + (int)((__brev((unsigned)e) >> 27) << (LOGN - 5))];
                        if (CHK) wide |= W::out_of_range(av[e], c);
                    }
                    // the row is in registers: its buffer takes the next column of the same parity before the arithmetic;
                    // past the end of the output row S takes column 0 of the next output row (or of the warp's next
                    // instances), X waits for the inverse transform below
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (j + 2 < l) fetch_a(base, i * l + j + 2, which);
                        else if (!which) {
                            if (i + 1 < k) fetch_a(base, (i + 1) * l, 0);
                            else if (nbase < count) fetch_a(nbase, 0, 0);
                        }
                    }
                } else {
                    const int32_t *arow = A + (((SHARED_A ? (size_t)0 : irow * k) + i) * l + j) * N + taurev;
#pragma unroll
                    for (int e = 0; e < 32; e++) {
                        av[e] = __ldg(arow + (int)((__brev((unsigned)e) >> 27) << (LOGN - 5)));
                        if (CHK) wide |= W::out_of_range(av[e], c);
                    }
                }
                // A is canonical in the reference (sampled in [0, q)); anything else is reduced first
                if (CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                    for (int e = 0; e < 32; e++) av[e] = W::bred(av[e], c);
                }
                const int32_t *sp = dyn_tiles + ((size_t)(j + 1) * C::POLYS + slot) * C::TS + 36 * tau;
#pragma unroll
                for (int e = 0; e < 32; e += 4) {
                    const int4 sv = *reinterpret_cast<const int4 *>(sp + e);
                    AR::acc_add(part[e], av[e], sv.x, c.k);
                    AR::acc_add(part[e + 1], av[e + 1], sv.y, c.k);
                    AR::acc_add(part[e + 2], av[e + 2], sv.z, c.k);
                    AR::acc_add(part[e + 3], av[e + 3], sv.w, c.k);
                }
            }
            u32 acc[NSUB][SUB];
#pragma unroll
            for (int e = 0; e < 32; e++) acc[e / SUB][e % SUB] = AR::acc_fin(part[e], c.k);
            if (TMA && i == k - 1) {
                // the stash is dead: the next instances' s rows travel during the last inverse transform
                fence_proxy_async();
                __syncwarp();
                if (lane == 0 && nbase < count) fetch_s(nbase);
            }
#pragma unroll
            for (int h = 0; h < NSUB; h++) {
                W::template inv_stages1<LOGN, LOGN - 1>(acc[h], c, tau, h);
                store_sub<SUB>(xt + 36 * tau + SUB * h, acc[h]);
            }
            __syncwarp();
            {
                u32 x[32];
                load_pass0<LOGN>(xt, x, tau);
                if (c.r0 & 1) {
#pragma unroll
                    for (int m = 0; m < 32; m++) x[m] = AR::red(x[m], c.one, c.k);
                }
                W::inv_pass0(x, c);
                if (ADD) W::template add_addend<LOGN, CHK>(x, e + (irow * k + i) * N, tau, c);
                if (live) {
                    int32_t *orow = out + (inst * k + i) * N;
#pragma unroll
                    for (int m = 0; m < 32; m++) orow[tau + m * T] = (int32_t)x[m];
                }
            }
            if (TMA && l >= 2) {
                // the exchange tile is free again: column 1 of the next output row (or of the next instances) into X
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    if (i + 1 < k) fetch_a(base, (i + 1) * l + 1, 1);
                    else if (nbase < count) fetch_a(nbase, 1, 1);
                }
            } else {
                __syncwarp();
            }
        }
        cl.advance(ctr);
    }
}


// ---- one matrix for the whole launch (scgpu_matvec_shared_batch) --------------------------------------------------
// With SHARED_A, k_matvec_rows_w32 and k_matvec16_w32 take the matrix from a table that k_matrix_table writes once per
// launch: every coefficient reduced to its centred residue (|a| <= q/2, inside every range window, so the kernels drop
// the range vote on it), each of the k l rows in thread-major order.  128-bit word v of thread tau of row r sits at
// (r V + v) T + tau and holds the thread's elements e = EW v .. EW v + EW - 1 (EW = 16 / sizeof(TE), V = 32 / EW), so
// for a fixed v the lanes of an instance read T consecutive 16-byte words -- the layout of the pass-1 twiddle tables.
// The table (8-16 KiB at Kyber's int16, up to 30 KiB at Dilithium's int32) stays in L1 / L2: only the s rows come from
// HBM.  The AR parameter only keeps the instantiations of the two policies' translation units apart.
template <class AR, class TE>
__global__ void k_matrix_table(TE *__restrict__ tab, const int32_t *__restrict__ A, int rows, int32_t q)
{
    using C = Cfg32<8>;
    constexpr int EW = 16 / (int)sizeof(TE), V = 32 / EW;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows * V * C::T) return;
    const int tau = t % C::T, v = (t / C::T) % V, r = t / (C::T * V);
    const int taurev = (int)(__brev((unsigned)tau) >> (32 - 3));
    alignas(16) TE w[EW];
#pragma unroll
    for (int u = 0; u < EW; u++) {
        const int e = v * EW + u;
        int32_t x = A[(size_t)r * C::N + taurev + (int)((__brev((unsigned)e) >> 27) << 3)] % q;
        if (x < 0) x += q;
        if (x > q / 2) x -= q;
        w[u] = (TE)x;
    }
    reinterpret_cast<int4 *>(tab)[t] = *reinterpret_cast<const int4 *>(w);
}

// the 32 elements of thread tau in row r of a k_matrix_table table (n = 256)
template <class TE>
__device__ __forceinline__ void load_table_row(int32_t (&av)[32], const int32_t *tab, int r, int tau)
{
    constexpr int T = Cfg32<8>::T, EW = 16 / (int)sizeof(TE), V = 32 / EW;
    const int4 *p = reinterpret_cast<const int4 *>(tab) + r * V * T + tau;
#pragma unroll
    for (int v = 0; v < V; v++) {
        const int4 w = __ldg(p + v * T);
        const int32_t wd[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int u = 0; u < 4; u++) {
            if constexpr (sizeof(TE) == 2) {
                av[8 * v + 2 * u] = (int32_t)(int16_t)(wd[u] & 0xFFFF);
                av[8 * v + 2 * u + 1] = wd[u] >> 16;
            } else {
                av[4 * v + u] = wd[u];
            }
        }
    }
}

// ---- mat-vec, one warp per OUTPUT ROW: the k warps of a CTA share the transformed vectors ------------------------
// k_matvec_w32 keeps l full 32-bit tiles per instance for ONE warp: 8 one-warp CTAs per SM at l = 4, two warps per
// scheduler, and the kernel is bound by fixed-latency dependencies (issue slots 41 % used, profiles/dil_matvec_r2g_ncu.json).
// Here a CTA of k warps works on the same PW instances: the forward transforms of the l vectors are split over the warps,
// a CTA barrier publishes the stash, then warp i accumulates and inverse-transforms output row i through its own
// exchange tile and staging row (two matrix rows in flight per warp, as above).  Shared memory per warp falls from
// l + 2 to l / k + 2 tiles: 15 warps per SM at k = 5, l = 4.  The s rows of the next group can only be requested after
// every warp has left the stash (second barrier); the matrix rows of the next group are requested before it.
// SHARED_A: the matrix is a k_matrix_table table (int32) read by 128-bit loads; no staging rows, no mbarrier per row.
// ADD: as in k_matvec_w32.
template <class AR, int LOGN, bool CHK = true, bool SHARED_A = false, bool ADD = false>
__global__ void __launch_bounds__(256, 2)
k_matvec_rows_w32(int32_t *__restrict__ out, const int32_t *__restrict__ A, const int32_t *__restrict__ s,
                  int k, int l, size_t count, unsigned long long *ctr, const __grid_constant__ W32Const<AR> c,
                  const int32_t *e)
{
    using C = Cfg32<LOGN>;
    using W = W32<AR>;
    constexpr int N = C::N, T = C::T, SUB = C::SUB, NSUB = C::NSUB, PW = C::PW;
    constexpr int AROW = N + T;
    constexpr int TILE = PW * C::TS;                                 // one tile per instance of the group
    constexpr int WARP_WORDS = SHARED_A ? TILE : TILE + PW * AROW;  // per warp: exchange tile (+ staging rows)
    constexpr uint32_t ROW_BYTES = (uint32_t)N * 4u;
    extern __shared__ __align__(16) int32_t dyn_tiles[];             // [l][PW][TS] stash | per warp: [PW][TS] | [PW][AROW]
    __shared__ __align__(8) uint64_t bar_s;                          // the s rows of a group (whole CTA)
    __shared__ __align__(8) uint64_t bars[8][2];                     // per warp: matrix rows in S, in X
    __shared__ unsigned s_next[2];                                   // the group after the next one, from the counter (by iteration parity)
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x / 32;
    const int nw = blockDim.x / 32;                                  // = k
    const int tau = lane % T;
    const int slot = lane / T;
    int32_t *mine = dyn_tiles + (size_t)l * TILE + (size_t)warp * WARP_WORDS;
    int32_t *xt = mine + slot * C::TS;
    const int32_t *astage = mine + TILE + slot * AROW;
    const int32_t *xstage = mine + slot * AROW;
    const int taurev = (int)(__brev((unsigned)tau) >> (32 - (LOGN - 5)));
    uint32_t par_s = 0, par_a0 = 0, par_a1 = 0;

    auto fetch_s = [&](size_t nbase) {                               // thread 0
        mbar_expect_tx(&bar_s, ROW_BYTES * PW * (uint32_t)l);
        for (int p = 0; p < PW; p++) {
            size_t row = nbase + p;
            if (row >= count) row = 0;
            for (int j = 0; j < l; j++)
                bulk_g2s(dyn_tiles + ((size_t)j * PW + p) * C::TS, s + (row * l + j) * N, ROW_BYTES, &bar_s);
        }
    };
    auto fetch_a = [&](size_t nbase, int step, int which) {          // lane 0 of the warp
        mbar_expect_tx(&bars[warp][which], ROW_BYTES * PW);
        int32_t *dst = which ? mine : mine + TILE;
        for (int p = 0; p < PW; p++) {
            size_t row = nbase + p;
            if (row >= count) row = 0;
            bulk_g2s(dst + p * AROW, A + (row * k * l + step) * N, ROW_BYTES, &bars[warp][which]);
        }
    };
    unsigned g = blockIdx.x, gn = blockIdx.x + gridDim.x, it = 0;
    if (threadIdx.x == 0) mbar_init(&bar_s, 1);
    if (lane == 0) {
        mbar_init(&bars[warp][0], 1);
        mbar_init(&bars[warp][1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if ((size_t)g * PW < count) {
        if (threadIdx.x == 0) fetch_s((size_t)g * PW);
        if (!SHARED_A && lane == 0) { fetch_a((size_t)g * PW, warp * l, 0); if (l >= 2) fetch_a((size_t)g * PW, warp * l + 1, 1); }
    }

    while ((size_t)g * PW < count) {
        const size_t base = (size_t)g * PW;
        const size_t nbase = (size_t)gn * PW;
        const size_t inst = base + slot;
        const bool live = inst < count;
        const int32_t *erow = e + ((live ? inst : 0) * k + warp) * N;     // this warp's output row i = warp
        if (ADD) prefetch_l2(erow + 32 * tau);
        // the group after the next one (read behind the second barrier of this iteration)
        if (threadIdx.x == 0)
            s_next[it & 1u] = ctr != nullptr ? atomicAdd(reinterpret_cast<unsigned *>(ctr), 1u) + 2u * gridDim.x : gn + gridDim.x;
        mbar_wait(&bar_s, par_s); par_s ^= 1u;
        // forward transforms of the vectors j = warp, warp + k, ... in place in their stash tiles
#pragma unroll 1
        for (int j = warp; j < l; j += nw) {
            int32_t *tile = dyn_tiles + ((size_t)j * PW + slot) * C::TS;
            {
                u32 x[32];
                W::template load_operand_staged<LOGN, CHK>(x, tile, tau, c);
                __syncwarp();
                W::fwd_pass0(x, c);
                store_pass0<LOGN>(tile, x, tau);
            }
            __syncwarp();
#pragma unroll 1
            for (int h = 0; h < NSUB; h++) {
                u32 xa[SUB], xb[SUB];
                int32_t *p = tile + 36 * tau + SUB * h;
                load_sub<SUB>(p, xa);
                W::template fwd_stages1<LOGN, C::S1, 1>(xa, xb, c, tau, h);
#pragma unroll
                for (int i = 0; i < SUB; i++) xa[i] = (u32)AR::dec(xa[i]);
                store_sub<SUB>(p, xa);                               // lane `lane` of every warp reads it back
            }
        }
        __syncthreads();                                             // the stash is complete
        {
            const int i = warp;                                      // this warp's output row
            typename AR::Acc part[32];
#pragma unroll
            for (int e = 0; e < 32; e++) part[e] = AR::acc_zero();
#pragma unroll 1
            for (int j = 0; j < l; j++) {
                int32_t av[32];
                bool wide = false;
                if constexpr (SHARED_A) {
                    load_table_row<int32_t>(av, A, i * l + j, tau);
                } else {
                    const int which = j & 1;
                    if (which) { mbar_wait(&bars[warp][1], par_a1); par_a1 ^= 1u; }
                    else       { mbar_wait(&bars[warp][0], par_a0); par_a0 ^= 1u; }
                    const int32_t *arow = which ? xstage : astage;
#pragma unroll
                    for (int e = 0; e < 32; e++) {
                        av[e] = arow[taurev + (int)((__brev((unsigned)e) >> 27) << (LOGN - 5))];
                        if (CHK) wide |= W::out_of_range(av[e], c);
                    }
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (j + 2 < l) fetch_a(base, i * l + j + 2, which);
                        else if (!which && nbase < count) fetch_a(nbase, i * l, 0);  // this warp's row of the next group
                    }
                }
                if (!SHARED_A && CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                    for (int e = 0; e < 32; e++) av[e] = W::bred(av[e], c);
                }
                const int32_t *sp = dyn_tiles + ((size_t)j * PW + slot) * C::TS + 36 * tau;
#pragma unroll
                for (int e = 0; e < 32; e += 4) {
                    const int4 sv = *reinterpret_cast<const int4 *>(sp + e);
                    AR::acc_add(part[e], av[e], sv.x, c.k);
                    AR::acc_add(part[e + 1], av[e + 1], sv.y, c.k);
                    AR::acc_add(part[e + 2], av[e + 2], sv.z, c.k);
                    AR::acc_add(part[e + 3], av[e + 3], sv.w, c.k);
                }
            }
            u32 acc[NSUB][SUB];
#pragma unroll
            for (int e = 0; e < 32; e++) acc[e / SUB][e % SUB] = AR::acc_fin(part[e], c.k);
            // this warp has left the stash: announce it before the inverse transform, which needs only the warp's own tile
            fence_proxy_async();
            __syncthreads();
            if (threadIdx.x == 0 && nbase < count) fetch_s(nbase);   // the next group's s rows travel during the inverse
#pragma unroll
            for (int h = 0; h < NSUB; h++) {
                W::template inv_stages1<LOGN, LOGN - 1>(acc[h], c, tau, h);
                store_sub<SUB>(xt + 36 * tau + SUB * h, acc[h]);
            }
            __syncwarp();
            {
                u32 x[32];
                load_pass0<LOGN>(xt, x, tau);
                if (c.r0 & 1) {
#pragma unroll
                    for (int m = 0; m < 32; m++) x[m] = AR::red(x[m], c.one, c.k);
                }
                W::inv_pass0(x, c);
                if (ADD) W::template add_addend<LOGN, CHK>(x, erow, tau, c);
                if (live) {
                    int32_t *orow = out + (inst * k + i) * N;
#pragma unroll
                    for (int m = 0; m < 32; m++) orow[tau + m * T] = (int32_t)x[m];
                }
            }
            if (!SHARED_A && l >= 2) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0 && nbase < count) fetch_a(nbase, i * l + 1, 1);
            } else {
                __syncwarp();
            }
        }
        g = gn;
        gn = *reinterpret_cast<volatile unsigned *>(&s_next[it & 1u]);   // written before the barriers of this iteration; the slot
        it++;                                                        // is rewritten two iterations (four barriers) later
    }
}


// ---- mat-vec with a 16-bit stash (moduli below 2^15.8, policies with AR::STASH16) --------------------------------
// The kernel above is limited to 8-9 warps per SM by the l full tiles it keeps per instance.  Here the transformed
// vectors are reduced to |x| <= q/2 + and kept as int16 (20 words per thread: conflict-free 128-bit reads), the
// forward transforms run through the one exchange tile, and EVERY row of the instance -- s_0 .. s_{l-1}, then
// A_00 .. A_{k-1,l-1} -- travels through ONE staging row and ONE mbarrier: as soon as a row is in registers the
// next row of the sequence (or s_0 of the warp's next instances) is put in flight.  13-15 warps per SM.
// IACC: the l products of an output coefficient cannot leave 32 bits (l |a| |s| < 2^31 with |a| <= x0 and the stash
// reduced to |s| <= 0.55 q), so they are summed by plain IMADs and the quotient comes from ONE conversion of the sum --
// instead of an IMAD, an FFMA and two conversions per term (AR::Acc), and in 32 instead of 64 accumulator registers.
// SHARED_A (with TMA): the matrix is a k_matrix_table table (int16) read by 128-bit loads; only the s rows travel
// through the staging row, and s_0 of the warp's next instances is put in flight as soon as s_{l-1} is in registers.
// ADD: as in k_matvec_w32.
template <class AR, int LOGN, bool TMA, bool CHK = true, bool IACC = false, bool SHARED_A = false, bool ADD = false>
__global__ void __launch_bounds__(kThreads32, 16)        // 128 registers: 4 warps per scheduler fit (140 allowed 3)
k_matvec16_w32(int32_t *__restrict__ out, const int32_t *__restrict__ A, const int32_t *__restrict__ s,
               int k, int l, size_t count, unsigned long long *ctr, const __grid_constant__ W32Const<AR> c,
               const int32_t *e)
{
    using C = Cfg32<LOGN>;
    using W = W32<AR>;
    constexpr int N = C::N, T = C::T, SUB = C::SUB, NSUB = C::NSUB;
    constexpr int AROW = N + T;                      // staging row stride: T banks between instances
    constexpr int SROW = 20 * T + T;                 // 16-bit stash row of one vector, in words (20 per thread)
    constexpr uint32_t ROW_BYTES = (uint32_t)N * 4u;
    extern __shared__ __align__(16) int32_t dyn_tiles[];             // [POLYS][TS] | [POLYS][AROW] | [l][POLYS][SROW]
    __shared__ __align__(8) uint64_t bars[kThreads32 / 32][2];       // [warp][0: rows through S, 1: rows through X]
    // this kernel sits at its register cap (128): the claimed group index lives in shared memory, and the claim is
    // made where it is first needed (when the last row of an instance has been consumed) instead of a whole
    // iteration ahead -- one exposed atomic per instance group (~1 % of its time)
    __shared__ unsigned s_gnext[kThreads32 / 32];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x / 32;
    const int tau = lane % T;
    const int slot = warp * C::PW + lane / T;
    int32_t *xt = dyn_tiles + slot * C::TS;
    int32_t *stage = dyn_tiles + C::POLYS * C::TS + slot * AROW;
    int32_t *stash0 = dyn_tiles + C::POLYS * (C::TS + AROW) + slot * SROW + 20 * tau;
    const int stash_stride = C::POLYS * SROW;                        // between vectors j
    const int taurev = (int)(__brev((unsigned)tau) >> (32 - (LOGN - 5)));
    // Rows travel through two buffers: S (the staging rows) takes the s rows and the even columns of the matrix, X (the
    // exchange tile, idle while an output row accumulates) the odd columns -- two matrix rows in flight per instance in
    // the same shared memory.  X is refilled only when the inverse transform (or, at the start of a group, the forward
    // transforms) has released the tile.
    const int32_t *xstage = dyn_tiles + slot * AROW;
    uint32_t par_s = 0, par_x = 0;

    // lane 0: row r of the sequence for the warp's PW instances starting at nbase
    auto fetch = [&](size_t nbase, int r, int which) {
        mbar_expect_tx(&bars[warp][which], ROW_BYTES * C::PW);
        int32_t *dst = which ? dyn_tiles : dyn_tiles + C::POLYS * C::TS;
        for (int p = 0; p < C::PW; p++) {
            size_t inst = nbase + (size_t)warp * C::PW + p;
            if (inst >= count) inst = 0;
            const int32_t *src = (SHARED_A || r < l) ? s + (inst * l + r) * N : A + (inst * k * l + (r - l)) * N;
            bulk_g2s(dst + (warp * C::PW + p) * AROW, src, ROW_BYTES, &bars[warp][which]);
        }
    };
    const size_t first = (size_t)blockIdx.x * C::POLYS;
    if (TMA) {
        if (lane == 0) {
            mbar_init(&bars[warp][0], 1);
            mbar_init(&bars[warp][1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        if (lane == 0 && first < count) fetch(first, 0, 0);
    }

    for (unsigned g = blockIdx.x; (size_t)g * C::POLYS < count;) {
        const size_t base = (size_t)g * C::POLYS;
        const size_t inst = base + slot;
        const bool live = inst < count;
        const size_t irow = live ? inst : 0;
        if (ADD) {
            for (int i = 0; i < k; i++) prefetch_l2(e + (irow * k + i) * N + 32 * tau);
        }
        // after a row of S has been read into registers: the next row of the S sequence (s rows, then the even columns
        // output row by output row), or row 0 of the warp's next instances; nxt = that row's number in the instance's
        // sequence (s rows 0 .. l-1, matrix rows l + i l + j), -1 = the instance has no further row for S
        auto advance_s = [&](int nxt) {
            if (TMA) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    if (nxt >= 0) fetch(base, nxt, 0);
                    else {
                        const unsigned gnext = claim_next(ctr, g, 0);
                        s_gnext[warp] = gnext;
                        const size_t nbase = (size_t)gnext * C::POLYS;
                        if (nbase < count) fetch(nbase, 0, 0);
                    }
                }
            }
        };
#pragma unroll 1
        for (int j = 0; j < l; j++) {
            u32 x[32];
            if (TMA) {
                mbar_wait(&bars[warp][0], par_s); par_s ^= 1u;
                W::template load_operand_staged<LOGN, CHK>(x, stage, tau, c);
                advance_s(SHARED_A && j + 1 == l ? -1 : j + 1);      // s row j + 1, or matrix row (0, 0) = number l
            } else {
                W::template load_operand<LOGN, CHK>(x, s + (irow * l + j) * N, tau, c);
            }
            W::fwd_pass0(x, c);
            store_pass0<LOGN>(xt, x, tau);
            __syncwarp();
#pragma unroll 1
            for (int h = 0; h < NSUB; h++) {
                u32 xa[SUB], xb[SUB];
                load_sub<SUB>(xt + 36 * tau + SUB * h, xa);
                W::template fwd_stages1<LOGN, C::S1, 1>(xa, xb, c, tau, h);
                // reduce, decode, pack two coefficients per word
                uint32_t pk[SUB / 2];
#pragma unroll
                for (int i = 0; i < SUB; i += 2) {
                    const int32_t v0 = AR::dec(AR::red(xa[i], c.one, c.k));
                    const int32_t v1 = AR::dec(AR::red(xa[i + 1], c.one, c.k));
                    pk[i / 2] = ((uint32_t)v0 & 0xFFFFu) | ((uint32_t)v1 << 16);
                }
                int32_t *dst = stash0 + j * stash_stride + (SUB / 2) * h;
#pragma unroll
                for (int i = 0; i < SUB / 2; i += 4)
                    *reinterpret_cast<uint4 *>(dst + i) = make_uint4(pk[i], pk[i + 1], pk[i + 2], pk[i + 3]);
            }
            __syncwarp();                                            // the exchange tile is reused by the next vector
        }
        if (!SHARED_A && TMA && l >= 2) {
            // the exchange tile is free until the first inverse transform: matrix row (0, 1) into X
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) fetch(base, l + 1, 1);
        }
#pragma unroll 1
        for (int i = 0; i < k; i++) {
            typename AR::Acc part[IACC ? 1 : 32];
            int32_t ipart[IACC ? 32 : 1];
#pragma unroll
            for (int e = 0; e < 32; e++) { if (IACC) ipart[e] = 0; else part[e] = AR::acc_zero(); }
#pragma unroll 1
            for (int j = 0; j < l; j++) {
                int32_t av[32];
                bool wide = false;
                if constexpr (SHARED_A) {
                    load_table_row<int16_t>(av, A, i * l + j, tau);
                } else if (TMA) {
                    const int which = j & 1;
                    if (which) { mbar_wait(&bars[warp][1], par_x); par_x ^= 1u; }
                    else       { mbar_wait(&bars[warp][0], par_s); par_s ^= 1u; }
                    const int32_t *arow = which ? xstage : stage;
#pragma unroll
                    for (int e = 0; e < 32; e++) {
                        av[e] = arow[taurev + (int)((__brev((unsigned)e) >> 27) << (LOGN - 5))];
                        if (CHK) wide |= W::out_of_range(av[e], c);
                    }
                    if (!which) {
                        advance_s(j + 2 < l ? l + i * l + j + 2 : (i + 1 < k ? l + (i + 1) * l : -1));
                    } else if (j + 2 < l) {
                        fence_proxy_async();
                        __syncwarp();
                        if (lane == 0) fetch(base, l + i * l + j + 2, 1);
                    }
                } else {
                    const int32_t *arow = A + ((irow * k + i) * l + j) * N + taurev;
#pragma unroll
                    for (int e = 0; e < 32; e++) {
                        av[e] = __ldg(arow + (int)((__brev((unsigned)e) >> 27) << (LOGN - 5)));
                        if (CHK) wide |= W::out_of_range(av[e], c);
                    }
                }
                if (!SHARED_A && CHK && __any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
                    for (int e = 0; e < 32; e++) av[e] = W::bred(av[e], c);
                }
                const int32_t *sp = stash0 + j * stash_stride;
#pragma unroll
                for (int e = 0; e < 32; e += 8) {
                    const uint4 sv = *reinterpret_cast<const uint4 *>(sp + e / 2);
                    const uint32_t wds[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int32_t s0 = (int32_t)(int16_t)(wds[u] & 0xFFFFu), s1 = (int32_t)wds[u] >> 16;
                        if constexpr (IACC) {
                            ipart[e + 2 * u] += av[e + 2 * u] * s0;
                            ipart[e + 2 * u + 1] += av[e + 2 * u + 1] * s1;
                        } else {
                            AR::acc_add(part[e + 2 * u], av[e + 2 * u], s0, c.k);
                            AR::acc_add(part[e + 2 * u + 1], av[e + 2 * u + 1], s1, c.k);
                        }
                    }
                }
            }
            u32 acc[NSUB][SUB];
#pragma unroll
            for (int e = 0; e < 32; e++) {
                if constexpr (IACC) acc[e / SUB][e % SUB] = AR::acc_fin_int(ipart[e], c.k);
                else acc[e / SUB][e % SUB] = AR::acc_fin(part[e], c.k);
            }
#pragma unroll
            for (int h = 0; h < NSUB; h++) {
                W::template inv_stages1<LOGN, LOGN - 1>(acc[h], c, tau, h);
                store_sub<SUB>(xt + 36 * tau + SUB * h, acc[h]);
            }
            __syncwarp();
            {
                u32 x[32];
                load_pass0<LOGN>(xt, x, tau);
                if (c.r0 & 1) {
#pragma unroll
                    for (int m = 0; m < 32; m++) x[m] = AR::red(x[m], c.one, c.k);
                }
                W::inv_pass0(x, c);
                if (ADD) W::template add_addend<LOGN, CHK>(x, e + (irow * k + i) * N, tau, c);
                if (live) {
                    int32_t *orow = out + (inst * k + i) * N;
#pragma unroll
                    for (int m = 0; m < 32; m++) orow[tau + m * T] = (int32_t)x[m];
                }
            }
            if (!SHARED_A && TMA && l >= 2 && i + 1 < k) {
                // the exchange tile is free again: column 1 of the next output row into X
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) fetch(base, l + (i + 1) * l + 1, 1);
            } else {
                __syncwarp();
            }
        }
        if (!TMA && lane == 0) s_gnext[warp] = claim_next(ctr, g, 0);
        __syncwarp();
        g = *reinterpret_cast<volatile unsigned *>(&s_gnext[warp]);
    }
}

// ---- host side, shared by the arithmetic policies -------------------------------------------------------------
// position of entry r (0 .. 16/len - 1) of thread tau in stage s of the thread-major pass-1 table
inline int slot32(int logn, int s, int tau, int r)
{
    const int n = 1 << logn, T = n / 32, len = n >> (s + 1), G = 16 / len, V = G < 4 ? G : 4;
    return (1 << s) + ((r / V) * T + tau) * V + (r % V);
}

// zf / zi: natural tables (index 2^s + b); returns [forward: WORDS arrays of n | inverse: WORDS arrays of n] with
// the entries of stages >= 5 in thread-major order.  get(e, k) = k-th 32-bit word of an entry.
template <class AR, class Vec, class Get>
inline void pack_pass1(int logn, const Vec &zf, const Vec &zi, Get get, int32_t *pack)
{
    const int n = 1 << logn, T = n / 32, W = AR::WORDS;
    for (int s = 5; s < logn; s++) {
        const int len = n >> (s + 1), G = 16 / len;
        for (int tau = 0; tau < T; tau++)
            for (int r = 0; r < G; r++) {
                const int nat = (1 << s) + tau * G + r, at = slot32(logn, s, tau, r);
                for (int k = 0; k < W; k++) {
                    pack[k * n + at] = get(zf[nat], k);
                    pack[(W + k) * n + at] = get(zi[nat], k);
                }
            }
    }
}

// group indices are 32-bit in the kernels (claim_next)
inline bool groups_fit(size_t groups, size_t grid) { return groups + 12 * grid < 0xFFFFFFFFull; }   // chunked claims overshoot by up to 2 chunks per warp

inline bool tma_allowed()
{
    const char *no_tma = getenv("SCGPU_NO_TMA");
    return !(no_tma && atoi(no_tma) != 0);
}

// Persistent grid over `count` rows in groups of per_group: min(SMs x per_sm, groups) CTAs; the groups after the first
// grid-full are claimed from a work counter, chunk groups per claim (*ctr stays nullptr when one grid-full holds them).
inline int persistent_grid(int sm_count, int per_sm, size_t count, int per_group, int chunk, cudaStream_t st,
                           unsigned *grid, unsigned long long **ctr)
{
    const size_t groups = (count + per_group - 1) / per_group;
    size_t g = (size_t)(sm_count > 0 ? sm_count : 148) * per_sm;
    if (g > groups) g = groups;
    if (!groups_fit(groups, g)) { set_error("batch of %zu rows is too large", count); return SCGPU_ERR_ARG; }
    *grid = (unsigned)g;
    *ctr = nullptr;
    return groups > g ? next_work_counter(st, ctr, chunk) : SCGPU_OK;
}

// bm: base-multiplication kernel (FQ_POLYMUL, policies with AR::BASEMUL; c must carry the (n/4)^-1 entries);
// chk = false: no range vote on the operands (nor on the addend); e != nullptr: out = (product + e) mod q
template <class AR>
int launch_polymul_w32(const W32Const<AR> &c, int logn, int sm_count, int mode, int32_t *out, const int32_t *a,
                       const void *b, size_t b_stride, size_t count, cudaStream_t st, bool bm = false, bool chk = true,
                       const int32_t *e = nullptr)
{
    // bulk copies need 16-byte aligned rows; the second operand is only staged in FQ_POLYMUL mode
    bool tma = ((uintptr_t)a % 16) == 0 && tma_allowed();
    if (mode == FQ_POLYMUL) tma = tma && ((uintptr_t)b % 16) == 0 && (b_stride % 4) == 0;
    if (mode == FQ_KEYBM && !(AR::BASEMUL && bm)) { set_error("key residue product: not available for this arithmetic"); return SCGPU_ERR_UNSUPPORTED; }
    if (mode != FQ_POLYMUL && mode != FQ_KEYBM) bm = false;
    if (!AR::BASEMUL) bm = false;
    if (logn < 8 || logn > 10) { set_error("unsupported n=%d", 1 << logn); return SCGPU_ERR_UNSUPPORTED; }
    return with_int<8, 9, 10>(logn, [&](auto L) {
        unsigned grid;
        unsigned long long *ctr;
        const int r = persistent_grid(sm_count, FQ32_MINB, count, Cfg32<L>::POLYS, 2, st, &grid, &ctr);
        if (r != SCGPU_OK) return r;
        return with_int<FQ_POLYMUL, FQ_KEY16, FQ_KEY32, FQ_KEYBM>(mode, [&](auto M) {
            return with_flags([&](auto TMA, auto BM, auto CHK, auto ADD) {
                // the base multiplication serves the two-operand product and is the only form of the residue product
                if constexpr ((BM ? AR::BASEMUL && (M == FQ_POLYMUL || M == FQ_KEYBM) : M != FQ_KEYBM) &&
                              AR::template serves<L, M, BM>())
                    return launch_kernel(k_polymul_w32<AR, L, M, TMA, BM, CHK, ADD>, grid, kThreads32, 0, st, out, a, b,
                                         b_stride, count, ctr, c, e);
                else
                    return SCGPU_ERR_UNSUPPORTED;
            }, tma, bm, chk, e != nullptr);
        });
    });
}

template <class AR>
int launch_ntt_w32(const W32Const<AR> &c, int logn, int sm_count, int inverse, int32_t *out, const int32_t *a, size_t count,
                   cudaStream_t st, bool chk = true)
{
    const bool tma = ((uintptr_t)a % 16) == 0 && tma_allowed();
    if (logn < 8 || logn > 10) { set_error("unsupported n=%d", 1 << logn); return SCGPU_ERR_UNSUPPORTED; }
    return with_int<8, 9, 10>(logn, [&](auto L) {
        unsigned grid;
        unsigned long long *ctr;
        const int e = persistent_grid(sm_count, FQ32_MINB, count, Cfg32<L>::POLYS, 2, st, &grid, &ctr);
        if (e != SCGPU_OK) return e;
        return with_flags([&](auto INV, auto TMA, auto CHK) {
            return launch_kernel(k_ntt_w32<AR, L, INV, TMA, CHK>, grid, kThreads32, 0, st, out, a, count, ctr, c);
        }, inverse != 0, tma, chk);
    });
}

// One shared matrix: its k_matrix_table table in a stream-ordered scratch of the call (not of the plan: two streams may
// run shared products with different matrices on one plan), written once before the batch kernel.
template <class AR, class TE>
int matrix_table(const W32Const<AR> &c, const int32_t *A, int rows, cudaStream_t st, int32_t **tab)
{
    const size_t words = (size_t)rows * Cfg32<8>::N * sizeof(TE) / 16;          // one thread per 128-bit word
    SCGPU_CUDA_CHECK(cudaMallocAsync(reinterpret_cast<void **>(tab), words * 16, st));
    const int e = launch_kernel(k_matrix_table<AR, TE>, (unsigned)((words + 127) / 128), 128, 0, st,
                                reinterpret_cast<TE *>(*tab), A, rows, c.q);
    if (e != SCGPU_OK) cudaFreeAsync(*tab, st);
    return e;
}

// the batch kernel has been launched (or refused, e != SCGPU_OK): release the table in stream order
inline int release_table(int32_t *tab, cudaStream_t st, int e)
{
    const cudaError_t fe = cudaFreeAsync(tab, st);
    if (e == SCGPU_OK && fe != cudaSuccess) { set_error("cudaFreeAsync failed: %s", cudaGetErrorString(fe)); return SCGPU_ERR_CUDA; }
    return e;
}

// n = 256 (Kyber, Dilithium).  shared: A is ONE matrix [k][l][n] for every instance (scgpu_matvec_shared_batch);
// e != nullptr: t = (product + e) mod q
template <class AR>
int launch_matvec_w32(const W32Const<AR> &c, int sm_count, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                      size_t count, cudaStream_t st, bool chk = true, bool shared = false, const int32_t *e = nullptr)
{
    using C = Cfg32<8>;
    const bool tma = ((uintptr_t)A % 16) == 0 && ((uintptr_t)s % 16) == 0 && tma_allowed();
    // the kernels below that read a shared matrix from its table stage only the s rows
    const bool tma_rows = shared ? ((uintptr_t)s % 16) == 0 && tma_allowed() : tma;
    unsigned grid;
    unsigned long long *ctr;
    int32_t *tab = nullptr;                          // the shared matrix's table
    // 16-bit stash: the reduced transform values must fit an int16 (|x| <= 0.55 q + 2)
    const char *no16 = getenv("SCGPU_MATVEC_STASH32");
    // measured (Kyber, q = 7681, tools/matvec_stash_ab.py): with the spill-free kernel the 16-bit stash wins for every l
    // (k = l = 2: 4.87 against 4.40e8 instances/s, k = 3, l = 2: 3.70 against 3.33e8, l = 3: equal); without bulk copies
    // the rows are not prefetched at all and the 32-bit stash kernel is used.  SCGPU_MATVEC16_MINL raises the threshold.
    const char *minl_env = getenv("SCGPU_MATVEC16_MINL");
    const int minl = minl_env ? atoi(minl_env) : 1;
    if (AR::STASH16 && c.q < 59000 && l >= minl && tma_rows && !(no16 && atoi(no16) != 0)) {
        const size_t smem = ((size_t)C::POLYS * (C::TS + (C::N + C::T)) + (size_t)l * C::POLYS * (20 * C::T + C::T)) * sizeof(int32_t);
        // integer accumulators: l |a| |s| < 2^31 with |a| <= x0 (the range vote's window, also what the flag promises) and
        // |s| <= 0.55 q + 2 (the reduced stash)
        const char *facc = getenv("SCGPU_MATVEC_FLOAT_ACC");
        const bool iacc = (double)l * (double)c.x0 * (0.55 * (double)c.q + 2.0) < 2147483648.0 && !(facc && atoi(facc) != 0);
        int per_sm = (int)((227 * 1024) / (smem + 1024 + 64));
        if (per_sm > 16) per_sm = 16;
        if (per_sm < 1) per_sm = 1;
        int r = persistent_grid(sm_count, per_sm, count, C::POLYS, 2, st, &grid, &ctr);
        // integer accumulators and shared matrices are instantiated for the policies with a 16-bit stash only
        if constexpr (AR::STASH16) {
            if (r == SCGPU_OK && shared) r = matrix_table<AR, int16_t>(c, A, k * l, st, &tab);
        }
        if (r != SCGPU_OK) return r;
        r = with_flags([&](auto CHK, auto IACC, auto SHARED, auto ADD) {
            if constexpr (AR::STASH16 || !(IACC || SHARED))
                return launch_kernel(k_matvec16_w32<AR, 8, true, CHK, IACC, SHARED, ADD>, grid, kThreads32, smem, st, out,
                                     shared ? tab : A, s, k, l, count, ctr, c, e);
            else
                return SCGPU_ERR_UNSUPPORTED;
        }, chk, iacc, shared, e != nullptr);
        return shared ? release_table(tab, st, r) : r;
    }
    // one warp per output row (k_matvec_rows_w32): aligned rows, 2 <= k <= 8; SCGPU_MATVEC_ONE_WARP=1 keeps k_matvec_w32.
    // A shared matrix needs no staging rows: each warp keeps only its exchange tile
    const char *ow = getenv("SCGPU_MATVEC_ONE_WARP");
    const size_t warp_words = shared ? (size_t)C::PW * C::TS : (size_t)C::PW * C::TS + C::PW * (C::N + C::T);
    const size_t smem_rows = ((size_t)l * C::PW * C::TS + (size_t)k * warp_words) * sizeof(int32_t);
    if (tma_rows && k >= 2 && k <= 8 && smem_rows <= 110 * 1024 && !(ow && atoi(ow) != 0)) {
        int per_sm = (int)((227 * 1024) / (smem_rows + 1024 + 256));
        const int by_regs = 65536 / (k * 32 * 128);
        if (per_sm > by_regs) per_sm = by_regs;
        if (per_sm < 1) per_sm = 1;
        int r = persistent_grid(sm_count, per_sm, count, C::PW, 1, st, &grid, &ctr);
        if (r == SCGPU_OK && shared) r = matrix_table<AR, int32_t>(c, A, k * l, st, &tab);
        if (r != SCGPU_OK) return r;
        r = with_flags([&](auto CHK, auto SHARED, auto ADD) {
            return launch_kernel(k_matvec_rows_w32<AR, 8, CHK, SHARED, ADD>, grid, 32 * k, smem_rows, st, out,
                                 shared ? tab : A, s, k, l, count, ctr, c, e);
        }, chk, shared, e != nullptr);
        return shared ? release_table(tab, st, r) : r;
    }
    // k = 1, unaligned rows, SCGPU_MATVEC_ONE_WARP: a shared matrix is addressed with an instance stride of 0
    const size_t smem = ((size_t)(l + 1) * C::POLYS * C::TS + (tma ? (size_t)C::POLYS * (C::N + C::T) : 0)) * sizeof(int32_t);
    if (smem > 200 * 1024) { set_error("matvec: l=%d needs %zu bytes of shared memory", l, smem); return SCGPU_ERR_UNSUPPORTED; }
    int per_sm = (int)((227 * 1024) / (smem + 1024 + 64));
    if (per_sm > 16) per_sm = 16;
    if (per_sm < 1) per_sm = 1;
    const int r = persistent_grid(sm_count, per_sm, count, C::POLYS, 2, st, &grid, &ctr);
    if (r != SCGPU_OK) return r;
    return with_flags([&](auto TMA, auto CHK, auto SHARED, auto ADD) {
        return launch_kernel(k_matvec_w32<AR, 8, TMA, CHK, SHARED, ADD>, grid, kThreads32, smem, st, out, A, s, k, l, count,
                             ctr, c, e);
    }, tma, chk, shared, e != nullptr);
}

}  // namespace w32
}  // namespace scgpu
