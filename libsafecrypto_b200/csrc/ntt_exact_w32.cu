// ntt_exact_w32.cu -- variant-exact fwd_ntt_32_16/32 and inv_ntt_32_16/32 on the warp-local 32-coefficient schedule.
//
// What the `*_32` table members return is the reference's lazily reduced, variant-specific representative
// (ntt_template.c.in:1541-1687): pre-twist by w, bit reversal, radix-2 DIT whose j = 0 column is never multiplied
// and whose sums are never reduced, post-twist by r and index flip for the inverse.  Every butterfly is an integer
// function of its two inputs, so ANY evaluation order of the same dataflow graph gives the reference's bits; the
// first version (ntt_exact.cu: k_transform) evaluated it with one butterfly per thread per stage and a shared-memory
// round trip + block barrier per stage, ~4500 warp-instructions per n = 512 transform (13 % of HBM peak).
//
// Here the same graph runs on the schedule of warp32.cuh.  The reference permutes, then runs a DIT; left in place
// on the UN-permuted array that DIT is: stage s pairs elements i, i + n / 2^(s+1) (top index bit first), the
// twiddle of the pair is w[brev_s(i >> (log n - s)) * n / 2^s], and element i ends up holding output brev(i).  So
//   pass 0  stages 0..4    thread tau holds elements tau + (n/32) m: all five stages are register-local and their 31
//                          twiddles are the same for every thread (constant bank), "j = 0" is a compile-time property
//                          of the register index;
//   pass 1  stages 5..     after ONE exchange through a padded tile the thread holds elements 32 tau .. 32 tau + 31;
//                          twiddles per thread from an L1-resident thread-major table; the j = 0 column only exists
//                          in thread 0;
//   output                 element e of thread tau is coefficient brev5(e) n/32 + brev(tau): for a fixed e the n/32
//                          lanes of a polynomial write n/32 consecutive words (whole sectors).
// n/32 threads per polynomial, polynomials never leave a warp (__syncwarp only), rows arrive by TMA bulk copy.
//
// Reductions, bit-exact per variant (reduce.cuh: Exact<V> remains the definition; the two cheap forms are proven
// equal to it below and compared with it -- and with the compiled reference -- over every test input):
//   reference   C `%` of the 64-bit product x w, sign of the dividend.  With the twiddle centred, wc = w or w - q,
//               and wp = round(wc 2^32 / q):  qe = hi32(x wp) = floor(x wc / q + eps), |eps| <= 1/4 for EVERY int32 x,
//               so t = x wc - qe q lies in (-q/4, 5q/4) and is congruent to x w.  Two unsigned-min steps bring
//               t - [x < 0] into [0, q); adding [x < 0] (1 - q) turns that into the remainder with the sign of x
//               (w > 0): 9 instructions, no 64-bit arithmetic, no bound on x.
//   barrett     ntt.c:366-378 literally, with the twiddle-times-m product precomputed: (x w) m == x (w m) mod 2^64,
//               w m < 2^30, so t = bits [k, k+32) of the 64-bit product x (w m): IMAD + IMAD.HI + funnel shift.
//   fp          (int64)(double(x w) * (1/q)) truncated, v - q qi (ntt_template.c.in:766-767).  With v = x w = m q + r:
//               the double product differs from v / q by less than 2^-21 (|v / q| < 2^31: 2^-22 from the rounded
//               reciprocal, 2^-23 from the product's own rounding), and r / q >= 1/q > 2^-21 for q < 2^21, so for
//               r != 0 the truncation is m and the result is the C remainder -- the reference variant's 9 instructions.
//               Only when q divides x w can the rounding fall below m (result q instead of 0, depending on q's
//               reciprocal and on m's position in its binade): that case -- one product in q -- takes the double
//               arithmetic itself.  For 32-bit tables (q up to 2^30) the bound needs |x| < 2^29; beyond it: doubles.
//   avx         scalar stages: the fp code.  Double lanes on 16-bit tables (|x w| < 2^46 < 2^51: the magic-number
//               conversion is exact): quotient = RN(x w (1/q)) in ONE rounding (FMA), and x w / q is never within
//               2^-21 of a half-integer (q odd), so the lane returns x w - round(x w / q) q, +q if negative: the
//               CANONICAL residue -- a Shoup product and two unsigned minima, no FP64.  Float lanes, full-range double
//               lanes (32-bit tables) and the q = 7681 twist stay lane emulation (Exact<V>).
//   solinas     Exact<V> as is (folds).
#include "warp32.cuh"

#include <cstring>
#include <vector>

namespace scgpu {

using namespace w32;

namespace {

struct XConst {
    const int32_t *p1;          // pass-1 twiddles: [w | aux], n words each, thread-major (slot32)
    const int32_t *tw;          // forward: pre-twist w[i]; inverse: post-twist r[k].  [w | aux], packed by 4 per thread
    int32_t f0w[31], f0a[31];   // stages 0..4: entry (1 << s) - 1 + g, g = m >> (5 - s)
    RedConst rc;
    int32_t nq, qm1;
    int32_t wp1;                // round(2^32 / q): the entry (1, wp1) turns ref_mul into x % q (modn of the integer fp form)
};

// position of word j (0..31) of thread t in the by-4 thread-major packing: a warp's 128-bit loads are contiguous
__host__ __device__ constexpr int by4(int T, int t, int j) { return ((j >> 2) * T + t) * 4 + (j & 3); }

// V_AVXF: the AVX2 variant with the single-precision lanes (16-bit tables, 512 < q <= 12289, ntt_template.c.in:1367-1402):
// a kernel of its own, so that no butterfly carries both lane flavours behind a run-time test of q
constexpr int V_AVXF = 6;
// Integer forms of the double arithmetic (file header), selected per plan (Xw32State::fpint: 16-bit tables, 0 <= w < q < 2^15,
// and no quotient m < 2^31 whose product m q rounds below m): fp, avx with double lanes, avx with float lanes
constexpr int V_FPI = 7, V_AVXI = 8, V_AVXFI = 9;
// 32-bit tables: the same integer forms hold while every multiplicand stays below 2^29 (and every lane product below
// 2^51), which a row guarantees when all its INPUTS are at most 2^27 (multiplicands are inputs, or sums of an input and
// a few residues below 2^26.4; twiddles are below 2^23.01).  V_FPG / V_AVXG vote on that per row; a row beyond the bound runs the double arithmetic over the same
// (centred) table entries, V_FPC / V_AVXC.
constexpr int V_FPG = 10, V_AVXG = 11, V_FPC = 12, V_AVXC = 13;
template <int V> struct PolicyOf {
    static constexpr int value = (V == V_AVXF || V == V_AVXI || V == V_AVXFI || V == V_AVXG || V == V_AVXC) ? (int)V_AVX
                               : ((V == V_FPI || V == V_FPG || V == V_FPC) ? (int)V_FP : V);
};
template <int V> constexpr bool kIntFp = (V == V_FPI || V == V_AVXI || V == V_AVXFI || V == V_FPG || V == V_AVXG);
template <int V> constexpr bool kFloatLanes = (V == V_AVXF || V == V_AVXFI);
template <int V> constexpr bool kGuarded = (V == V_FPG || V == V_AVXG);
template <int V> constexpr bool kCentredDoubles = (V == V_FPC || V == V_AVXC);       // doubles over (wc, wp) entries
template <int V> struct SlowOf { static constexpr int value = V == V_FPG ? V_FPC : (V == V_AVXG ? V_AVXC : V); };
template <int V> struct XTag { static constexpr int value = V; };

// C remainder of x * w (sign of x), w > 0 given centred with wp = round(wc 2^32 / q); any int32 x
__device__ __forceinline__ int32_t ref_mul(int32_t x, int32_t wc, int32_t wp, const XConst &c)
{
    const int32_t s = x >> 31;
    const int32_t qe = __mulhi(x, wp);
    const uint32_t p = (uint32_t)x * (uint32_t)wc + (uint32_t)s;
    uint32_t t = (uint32_t)qe * (uint32_t)c.nq + p;
    t = min(t, t + (uint32_t)c.rc.q);
    t = min(t, t - (uint32_t)c.rc.q);
    return (int32_t)((uint32_t)s * (uint32_t)c.qm1 + t);
}
// canonical residue of x * w in [0, q), same entry
__device__ __forceinline__ int32_t canon_mul(int32_t x, int32_t wc, int32_t wp, const XConst &c)
{
    const int32_t qe = __mulhi(x, wp);
    uint32_t t = (uint32_t)x * (uint32_t)wc + (uint32_t)qe * (uint32_t)c.nq;        // in (-q/4, 5q/4)
    t = min(t, t + (uint32_t)c.rc.q);
    t = min(t, t - (uint32_t)c.rc.q);
    return (int32_t)t;
}

template <int V, bool TW16>
__device__ __forceinline__ int32_t xmul(int32_t x, int32_t w, int32_t aux, const XConst &c)
{
    constexpr int EV = PolicyOf<V>::value;
    if constexpr (V == V_REFERENCE) {
        return ref_mul(x, w, aux, c);                                               // w is the centred twiddle here
    } else if constexpr (V == V_BARRETT) {
        const uint32_t lo = (uint32_t)x * (uint32_t)aux;                            // aux = w * m
        const uint32_t hi = (uint32_t)__mulhi(x, aux);
        const uint32_t t = __funnelshift_r(lo, hi, c.rc.k);
        const uint32_t v = (uint32_t)x * (uint32_t)w + t * (uint32_t)c.nq;
        return cond_fix((int32_t)v, c.rc.q);
    } else if constexpr (kIntFp<V>) {
        // fp and the scalar stages of avx where the truncated double quotient provably IS the C remainder (file header):
        // entries are (wc, wp) as for the reference variant
        return ref_mul(x, w, aux, c);
    } else {
        // fp and the scalar stages of avx otherwise: the double quotient with its two 64-bit conversions.  A
        // conversion-free form (magic-number int -> double and truncation) was measured SLOWER: it trades two XU
        // conversions for five more FP64-pipe operations (fp forward n = 512: 7.5e8 -> 5.3e8 transforms/s).
        return Exact<EV>::muln(x, kCentredDoubles<V> ? w + ((w >> 31) & c.rc.q) : w, c.rc);
    }
}

// pointwise twist element: mul_32_pointwise(_16) of the variant (the AVX2 build runs its vector lanes here)
template <int V, bool TW16>
__device__ __forceinline__ int32_t xtwist(int32_t x, int32_t w, int32_t aux, const XConst &c)
{
    constexpr int EV = PolicyOf<V>::value;
    if constexpr (EV == V_AVX) {
        if constexpr (kIntFp<V>) return canon_mul(x, w, aux, c);       // double lane (16-bit tables with q != 7681, guarded rows of 32-bit tables): canonical residue
        else {
            const int32_t wu = kCentredDoubles<V> ? w + ((w >> 31) & c.rc.q) : w;
            return TW16 ? Exact<EV>::pw16(x, wu, c.rc) : Exact<EV>::pw32(x, wu, c.rc);
        }
    } else {
        return xmul<V, TW16>(x, w, aux, c);
    }
}

// one DIT butterfly of stage S (ntt_template.c.in:1144-1244 fft_32, :1341-1482 fft_16; the AVX2 branches
// :1164-1203 / :1361-1438 run the vector lanes on every column of the stages with half < n/8)
template <int V, int LOGN, int S, bool TW16>
__device__ __forceinline__ void xbfly(int32_t &lo, int32_t &hi, int32_t w, int32_t aux, bool j0, const XConst &c)
{
    constexpr int N = 1 << LOGN;
    constexpr int EV = PolicyOf<V>::value;
    constexpr bool vec = (EV == V_AVX) && ((1 << S) < (N >> 3));
    int32_t x;
    if constexpr (vec) {
        if constexpr (kFloatLanes<V>)  x = lane_flt_magic((int32_t)((uint32_t)hi * (uint32_t)w), c.rc);   // low 32 bits of the product
        else if constexpr (kIntFp<V>)  x = canon_mul(hi, w, aux, c);                                      // double lane, 16-bit tables
        else                           x = lane_dbl((int64_t)hi * (int64_t)(kCentredDoubles<V> ? w + ((w >> 31) & c.rc.q) : w), false, c.rc);
    } else {
        // column j = 0 is not multiplied: passed through (fft_16) or reduced only (fft_32); the integer fp form of
        // modn is the remainder x % q (|x| / q < 2^9: no bound on x is needed)
        int32_t x0;
        if constexpr (TW16) x0 = hi;
        else if constexpr (kIntFp<V>) x0 = ref_mul(hi, 1, c.wp1, c);
        else x0 = Exact<EV>::modn(hi, c.rc);
        if (S == 0) x = x0;
        else {
            const int32_t xm = xmul<V, TW16>(hi, w, aux, c);
            x = j0 ? x0 : xm;
        }
    }
    hi = (int32_t)((uint32_t)lo - (uint32_t)x);
    lo = (int32_t)((uint32_t)lo + (uint32_t)x);
}

template <int V, int LOGN, bool TW16>
__device__ __forceinline__ void xpass0(int32_t (&x)[32], const XConst &c)
{
#pragma unroll
    for (int s = 0; s < 5; s++) {
        const int half = 16 >> s;
#pragma unroll
        for (int m = 0; m < 32; m++)
            if ((m & half) == 0) {
                const int g = m >> (5 - s);
                const int idx = (1 << s) - 1 + g;
                // s is a compile-time constant after unrolling; dispatch on it for the stage template parameter
                if (s == 0)      xbfly<V, LOGN, 0, TW16>(x[m], x[m + half], c.f0w[idx], c.f0a[idx], g == 0, c);
                else if (s == 1) xbfly<V, LOGN, 1, TW16>(x[m], x[m + half], c.f0w[idx], c.f0a[idx], g == 0, c);
                else if (s == 2) xbfly<V, LOGN, 2, TW16>(x[m], x[m + half], c.f0w[idx], c.f0a[idx], g == 0, c);
                else if (s == 3) xbfly<V, LOGN, 3, TW16>(x[m], x[m + half], c.f0w[idx], c.f0a[idx], g == 0, c);
                else             xbfly<V, LOGN, 4, TW16>(x[m], x[m + half], c.f0w[idx], c.f0a[idx], g == 0, c);
            }
    }
}

// CNT consecutive pass-1 entries r0 .. r0 + CNT - 1 of thread tau for stage S (same table layout as W32::load_entries)
template <int LOGN, int S, int CNT>
__device__ __forceinline__ void xload_entries(int32_t (&w)[CNT], int32_t (&a)[CNT], const int32_t *tab, int tau, int r0)
{
    using C = Cfg32<LOGN>;
    constexpr int LEN = C::N >> (S + 1);
    constexpr int G = 16 / LEN;
    constexpr int Vv = G < 4 ? G : 4;
    const int32_t *p = tab + (1 << S) + ((r0 / Vv) * C::T + tau) * Vv + (r0 % Vv);
    if constexpr (CNT == 4) {
        const int4 v0 = __ldg(reinterpret_cast<const int4 *>(p)), v1 = __ldg(reinterpret_cast<const int4 *>(p + C::N));
        w[0] = v0.x; w[1] = v0.y; w[2] = v0.z; w[3] = v0.w;
        a[0] = v1.x; a[1] = v1.y; a[2] = v1.z; a[3] = v1.w;
    } else if constexpr (CNT == 2) {
        const int2 v0 = __ldg(reinterpret_cast<const int2 *>(p)), v1 = __ldg(reinterpret_cast<const int2 *>(p + C::N));
        w[0] = v0.x; w[1] = v0.y; a[0] = v1.x; a[1] = v1.y;
    } else {
        w[0] = __ldg(p); a[0] = __ldg(p + C::N);
    }
}

template <int V, int LOGN, int S, bool TW16>
__device__ __forceinline__ void xstage1(int32_t (&x)[32], const XConst &c, int tau)
{
    using C = Cfg32<LOGN>;
    constexpr int LEN = C::N >> (S + 1);
    constexpr int CNT = 32 / (2 * LEN);
    constexpr int GRP = CNT < 4 ? CNT : 4;
#pragma unroll
    for (int g0 = 0; g0 < CNT; g0 += GRP) {
        int32_t w[GRP], a[GRP];
        xload_entries<LOGN, S, GRP>(w, a, c.p1, tau, g0);
#pragma unroll
        for (int g = 0; g < GRP; g++) {
            const bool j0 = (g0 + g == 0) && tau == 0;            // group index tau * CNT + g0 + g == 0
#pragma unroll
            for (int j = 0; j < LEN; j++) {
                const int i = (g0 + g) * 2 * LEN + j;
                xbfly<V, LOGN, S, TW16>(x[i], x[i + LEN], w[g], a[g], (g0 + g == 0) ? j0 : false, c);
            }
        }
    }
}
template <int V, int LOGN, int S, bool TW16>
__device__ __forceinline__ void xstages1(int32_t (&x)[32], const XConst &c, int tau)
{
    if constexpr (S < LOGN) {
        xstage1<V, LOGN, S, TW16>(x, c, tau);
        xstages1<V, LOGN, S + 1, TW16>(x, c, tau);
    }
}

template <int V, int LOGN, bool TW16, bool INV, bool TMA>
__global__ void __launch_bounds__(kThreads32, 16)
k_exact_w32(int32_t *__restrict__ out, const int32_t *__restrict__ a, size_t count, unsigned long long *ctr,
            const __grid_constant__ XConst c)
{
    using C = Cfg32<LOGN>;
    constexpr int N = C::N, T = C::T;
    constexpr int AROW = N + T;
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
    uint32_t parity = 0;
    auto fetch = [&](size_t nbase) {
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

    w32::Claim cl;
    for (cl.init(ctr, (unsigned)((count + C::POLYS - 1) / C::POLYS)); (size_t)cl.g * C::POLYS < count;) {
        const size_t base = (size_t)cl.g * C::POLYS;
        const size_t poly = base + slot;
        const bool live = poly < count;
        const size_t prow = live ? poly : 0;
        cl.issue(ctr, lane);
        const size_t nbase = (size_t)cl.gn * C::POLYS;
        int32_t xr[32];                                             // the raw row
        {
            if (TMA) {
                mbar_wait(&bars[warp], parity); parity ^= 1u;
#pragma unroll
                for (int m = 0; m < 32; m++) xr[m] = stage[tau + m * T];
                fence_proxy_async();
                __syncwarp();
                if (lane == 0 && nbase < count) fetch(nbase);        // the staging row is in registers
            } else {
#pragma unroll
                for (int m = 0; m < 32; m++) xr[m] = __ldg(a + prow * N + tau + m * T);
            }
        }
        auto row_body = [&](auto tag) {
        constexpr int VV = decltype(tag)::value;
        {
            int32_t x[32];
#pragma unroll
            for (int m = 0; m < 32; m++) x[m] = xr[m];
            if (!INV) {
                // pre-twist v[i] = t[i] * w[i], i = tau + T m (mult_pointwise, :956-1141)
#pragma unroll
                for (int m4 = 0; m4 < 32; m4 += 4) {
                    const int4 w4 = __ldg(reinterpret_cast<const int4 *>(c.tw + by4(T, tau, m4)));
                    const int4 a4 = __ldg(reinterpret_cast<const int4 *>(c.tw + N + by4(T, tau, m4)));
                    x[m4] = xtwist<VV, TW16>(x[m4], w4.x, a4.x, c);
                    x[m4 + 1] = xtwist<VV, TW16>(x[m4 + 1], w4.y, a4.y, c);
                    x[m4 + 2] = xtwist<VV, TW16>(x[m4 + 2], w4.z, a4.z, c);
                    x[m4 + 3] = xtwist<VV, TW16>(x[m4 + 3], w4.w, a4.w, c);
                }
            }
            xpass0<VV, LOGN, TW16>(x, c);
#pragma unroll
            for (int m = 0; m < 32; m++) tile[tau + pos32(T * m)] = x[m];
        }
        __syncwarp();
        {
            int32_t x[32];
#pragma unroll
            for (int k4 = 0; k4 < 32; k4 += 4) {
                const int4 v = *reinterpret_cast<const int4 *>(tile + 36 * tau + k4);
                x[k4] = v.x; x[k4 + 1] = v.y; x[k4 + 2] = v.z; x[k4 + 3] = v.w;
            }
            xstages1<VV, LOGN, 5, TW16>(x, c, tau);
            if (!INV) {
                if (live) {
                    int32_t *orow = out + poly * N + ntt_index<LOGN>(tau, 0);
#pragma unroll
                    for (int e = 0; e < 32; e++) orow[(int)((__brev((unsigned)e) >> 27) << (LOGN - 5))] = x[e];
                }
            } else {
                // post-twist by r, then ntt32_flip_generic (ntt.c:571-604): out[i] = fix(i ? v'[n - i] : -v'[0])
                const int k0 = ntt_index<LOGN>(tau, 0);                              // coefficient index of element 0
#pragma unroll
                for (int e4 = 0; e4 < 32; e4 += 4) {
                    const int4 w4 = __ldg(reinterpret_cast<const int4 *>(c.tw + by4(T, tau, e4)));
                    const int4 a4 = __ldg(reinterpret_cast<const int4 *>(c.tw + N + by4(T, tau, e4)));
                    const int32_t ws[4] = {w4.x, w4.y, w4.z, w4.w}, as[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e4 + u;
                        const int k = k0 + (int)((__brev((unsigned)e) >> 27) << (LOGN - 5));
                        int32_t v;
                        if constexpr (VV == V_REFERENCE || kIntFp<VV>) {
                            // cond_fix of the C remainder (and of the double lane's residue) IS the canonical residue:
                            // one Shoup product and two minima instead of remainder + sign + fix-up; -v for k = 0
                            v = canon_mul(x[e], ws[u], as[u], c);
                            if (e == 0) v = (k == 0 && v != 0) ? c.rc.q - v : v;
                        } else {
                            v = xtwist<VV, TW16>(x[e], ws[u], as[u], c);
                            if (e == 0) v = (k == 0) ? (int32_t)(0u - (uint32_t)v) : v;
                            v = cond_fix(v, c.rc.q);
                        }
                        if (live) out[poly * N + ((N - k) & (N - 1))] = v;
                    }
                }
            }
        }
        };
        if constexpr (kGuarded<V>) {
            bool big = false;
#pragma unroll
            for (int m = 0; m < 32; m++) big |= ((uint32_t)xr[m] + 0x08000000u) > 0x10000000u;      // |input| > 2^27
            if (__any_sync(0xFFFFFFFFu, big)) row_body(XTag<SlowOf<V>::value>{});
            else row_body(XTag<V>{});
        } else {
            row_body(XTag<V>{});
        }
        __syncwarp();
        cl.advance(ctr);
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------

struct ArX { static constexpr int WORDS = 2; };       // two words per entry for pack_pass1

int32_t centre(int32_t w, int32_t q) { return w > q / 2 ? w - q : w; }

// the two words of a twiddle entry for the plan's variant.  kind: 0 = stage with the AVX2 vector lanes (avx only),
// 1 = scalar stage, 2 = pre / post twist
void make_entry(const NttPlanDev &p, bool fpint, int32_t w, int kind, int32_t *ow, int32_t *oa)
{
    const int32_t q = p.rc.q;
    const bool tw16 = p.tw_bits == 16;
    bool centred = false;
    if (p.variant == V_REFERENCE) centred = true;
    else if (p.variant == V_FP) centred = fpint;
    else if (p.variant == V_AVX && fpint) {
        const bool avxf = tw16 && q <= 12289;                    // float lanes in the vector stages
        if (kind == 0) centred = !avxf;                          // double lanes: canonical Shoup product
        else if (kind == 1) centred = true;                      // fp code
        else centred = !tw16 || q != 7681;                       // twist: double lanes unless 16-bit tables with q = 7681 (float lanes)
    }
    if (centred) {
        const int32_t wc = centre(w, q);
        const double wp = nearbyint((double)wc * 4294967296.0 / (double)q);           // |wp| < 2^31
        *ow = wc;
        *oa = (int32_t)(int64_t)wp;
    } else if (p.variant == V_BARRETT) {
        *ow = w;
        *oa = (int32_t)((int64_t)w * (int64_t)p.rc.m);
    } else {
        *ow = w;
        *oa = 0;
    }
}

}  // namespace

struct Xw32State {
    int32_t *tab;                        // [pass-1 w | aux | fwd twist w | aux | inv twist w | aux], n words each
    bool inverse;                        // r given: inverse transforms too
    bool fpint;                          // fp / avx: the double quotient is evaluated in integers (file header)
    XConst fwd, inv;
};

// Eligibility and tables.  reference / barrett need canonical twiddles 0 <= w < q (the sign of the remainder follows
// the dividend only then; every table the reference generates qualifies) and, for barrett, k in [0, 31] with
// w * m inside 32 bits; anything else stays on the first kernel.
int build_xw32_tables(NttPlanDev &p, const int32_t *w_host, const int32_t *r_host)
{
    if (p.logn < 8 || p.logn > 10 || !w_host) return SCGPU_OK;
    const int n = p.n, L = p.logn, T = n / 32;
    const int32_t q = p.rc.q;
    if (q < 3 || q >= (1 << 30)) return SCGPU_OK;
    bool fpint = false;
    bool canonical = true;
    for (int i = 0; i < n; i++) {
        if (w_host[i] < 0 || w_host[i] >= q) canonical = false;
        if (r_host && (r_host[i] < 0 || r_host[i] >= q)) canonical = false;
    }
    if (p.variant == V_REFERENCE || p.variant == V_BARRETT) {
        if (!canonical) return SCGPU_OK;
        if (p.variant == V_BARRETT) {
            if (p.rc.k < 0 || p.rc.k > 31 || p.rc.m < 0) return SCGPU_OK;
            if ((int64_t)(q - 1) * (int64_t)p.rc.m > 0x7FFFFFFFll) return SCGPU_OK;
        }
    }
    if ((p.variant == V_FP || p.variant == V_AVX) && canonical && (q & 1) &&
        ((p.tw_bits == 16 && q < (1 << 15)) || (p.tw_bits != 16 && q < 8400000))) {
        // (32-bit tables: rows are guarded, see V_FPG; q < 2^23.002 keeps the guarded bounds -- quotient error
        // 1.5 * 2^-25.3 below 1/q, lane products below 2^51)
        // Integer forms (file header).  The truncated quotient of an exact multiple m q is m unless RN(m (1 + delta)) < m,
        // delta = inv_q_dbl q - 1 (the caller's reciprocal, not recomputed): impossible for delta >= 0, and for delta < 0
        // only when m |delta| exceeds half the spacing below m, i.e. (m / 2^k) |delta| 2^53 > 1 with m / 2^k < 2.
        const long double delta = (long double)p.rc.inv_q_dbl * (long double)q - 1.0L;      // exact: 53 + 15 bits < 64
        const long double D = -delta * 9007199254740992.0L;                                  // |delta| 2^53 when delta < 0
        if (delta >= 0.0L || D <= 0.5L) fpint = true;
        if (p.variant == V_AVX && q == 7681) fpint = false;      // its twist runs the float lanes (mul_32_pointwise_16, :1081-1094)
    }
    auto brev_bits = [](int v, int bits) { int r = 0; for (int b = 0; b < bits; b++) if (v & (1 << b)) r |= 1 << (bits - 1 - b); return r; };
    // natural table: entry 2^s + g = w[brev_s(g) * n / 2^s]
    struct Ent { int32_t w, a; };
    std::vector<Ent> z(n), zdummy(n);
    for (int s = 0; s < L; s++)
        for (int g = 0; g < (1 << s); g++) {
            Ent e;
            const int vec = (p.variant == V_AVX && (1 << s) < (n >> 3)) ? 0 : 1;       // ntt_template.c.in:1164, :1361
            make_entry(p, fpint, w_host[(size_t)brev_bits(g, s) << (L - s)], vec, &e.w, &e.a);
            z[(1 << s) + g] = e;
        }
    // layout: [pass-1 w | pass-1 aux | fwd twist w | fwd twist aux | inv twist w | inv twist aux], n words each
    std::vector<int32_t> pack(6 * (size_t)n, 0);
    std::vector<int32_t> p1(4 * (size_t)n, 0);
    pack_pass1<ArX>(L, z, zdummy, [](const Ent &e, int k) { return k == 0 ? e.w : e.a; }, p1.data());
    memcpy(pack.data(), p1.data(), sizeof(int32_t) * 2 * n);
    for (int t = 0; t < T; t++)
        for (int j = 0; j < 32; j++) {
            int32_t ew, ea;
            make_entry(p, fpint, w_host[t + T * j], 2, &ew, &ea);                            // pre-twist of element tau + T m
            pack[2 * n + by4(T, t, j)] = ew; pack[3 * n + by4(T, t, j)] = ea;
            if (r_host) {
                const int k = (brev_bits(j, 5) << (L - 5)) | brev_bits(t, L - 5);      // coefficient of element j, thread t
                make_entry(p, fpint, r_host[k], 2, &ew, &ea);
                pack[4 * n + by4(T, t, j)] = ew; pack[5 * n + by4(T, t, j)] = ea;
            }
        }
    Xw32State *xs = p.xw32 = new Xw32State();
    xs->inverse = r_host != nullptr;
    xs->fpint = fpint;
    SCGPU_CUDA_CHECK(cudaMalloc(&xs->tab, sizeof(int32_t) * pack.size()));
    SCGPU_CUDA_CHECK(cudaMemcpy(xs->tab, pack.data(), sizeof(int32_t) * pack.size(), cudaMemcpyHostToDevice));
    XConst c;
    c.p1 = xs->tab;
    for (int i = 0; i < 31; i++) { c.f0w[i] = z[i + 1].w; c.f0a[i] = z[i + 1].a; }
    c.rc = p.rc;
    c.nq = -q;
    c.qm1 = q - 1;
    c.wp1 = (int32_t)(int64_t)nearbyint(4294967296.0 / (double)q);
    xs->fwd = xs->inv = c;
    xs->fwd.tw = xs->tab + 2 * (size_t)n;
    xs->inv.tw = xs->tab + 4 * (size_t)n;
    return SCGPU_OK;
}

void free_xw32_tables(NttPlanDev &p)
{
    if (!p.xw32) return;
    cudaFree(p.xw32->tab);
    delete p.xw32;
    p.xw32 = nullptr;
}

namespace {

template <int V, int LOGN, bool TW16>
int launch_x(const NttPlanDev &p, bool inverse, int32_t *out, const int32_t *a, size_t count, const XConst &c, cudaStream_t st)
{
    // rows that are not 16-byte aligned cannot be bulk-copied: they stay on the first kernel
    if (((uintptr_t)a % 16) != 0 || !tma_allowed()) return SCGPU_ERR_UNSUPPORTED;
    unsigned grid;
    unsigned long long *ctr;
    const int e = persistent_grid(p.sm_count, 16, count, Cfg32<LOGN>::POLYS, 4, st, &grid, &ctr);
    if (e != SCGPU_OK) return e;
    if (inverse) return launch_kernel(k_exact_w32<V, LOGN, TW16, true, true>, grid, kThreads32, 0, st, out, a, count, ctr, c);
    return launch_kernel(k_exact_w32<V, LOGN, TW16, false, true>, grid, kThreads32, 0, st, out, a, count, ctr, c);
}

template <int V>
int launch_xv(const NttPlanDev &p, bool inverse, int32_t *out, const int32_t *a, size_t count, const XConst &c, cudaStream_t st)
{
    const bool tw16 = p.tw_bits == 16;
    if constexpr (V == V_SOL7681) {
        if (p.logn != 8 || !tw16) return SCGPU_ERR_UNSUPPORTED;
        return launch_x<V, 8, true>(p, inverse, out, a, count, c, st);
    } else if constexpr (V == V_SOL8380417) {
        if (p.logn != 8 || tw16) return SCGPU_ERR_UNSUPPORTED;
        return launch_x<V, 8, false>(p, inverse, out, a, count, c, st);
    } else if constexpr (kGuarded<V>) {
        if (tw16) return SCGPU_ERR_UNSUPPORTED;
        switch (p.logn) {
        case 8:  return launch_x<V, 8, false>(p, inverse, out, a, count, c, st);
        case 9:  return launch_x<V, 9, false>(p, inverse, out, a, count, c, st);
        case 10: return launch_x<V, 10, false>(p, inverse, out, a, count, c, st);
        default: return SCGPU_ERR_UNSUPPORTED;
        }
    } else if constexpr (V == V_AVXF || kIntFp<V>) {
        if (!tw16) return SCGPU_ERR_UNSUPPORTED;
        switch (p.logn) {
        case 8:  return launch_x<V, 8, true>(p, inverse, out, a, count, c, st);
        case 9:  return launch_x<V, 9, true>(p, inverse, out, a, count, c, st);
        case 10: return launch_x<V, 10, true>(p, inverse, out, a, count, c, st);
        default: return SCGPU_ERR_UNSUPPORTED;
        }
    } else
    // the parameter sets of the reference: 16-bit tables exist for n = 256 (7681), 512 / 1024 (12289, 18433);
    // 32-bit tables for n = 256 (8380417), 512, 1024
#ifndef XW32_LOGNS
#define XW32_LOGNS 7
#endif
    switch (p.logn) {
#if XW32_LOGNS & 1
    case 8:  return tw16 ? launch_x<V, 8, true>(p, inverse, out, a, count, c, st) : launch_x<V, 8, false>(p, inverse, out, a, count, c, st);
#endif
#if XW32_LOGNS & 2
    case 9:  return tw16 ? launch_x<V, 9, true>(p, inverse, out, a, count, c, st) : launch_x<V, 9, false>(p, inverse, out, a, count, c, st);
#endif
#if XW32_LOGNS & 4
    case 10: return tw16 ? launch_x<V, 10, true>(p, inverse, out, a, count, c, st) : launch_x<V, 10, false>(p, inverse, out, a, count, c, st);
#endif
    default: return SCGPU_ERR_UNSUPPORTED;
    }
}

}  // namespace

// SCGPU_ERR_UNSUPPORTED: the caller runs the first kernel (ntt_exact.cu)
int launch_exact_w32(const NttPlanDev &p, int op, int32_t *out, const int32_t *a, size_t count, cudaStream_t st)
{
    if (op != SCGPU_OP_FWD && op != SCGPU_OP_INV) return SCGPU_ERR_UNSUPPORTED;
    const bool inverse = op == SCGPU_OP_INV;
    if (!p.xw32 || (inverse && !p.xw32->inverse)) return SCGPU_ERR_UNSUPPORTED;
    if (out == a && count > 0) {
        // in place is fine: a row is read completely (into registers / the staging row) before any of it is written,
        // and rows are independent -- except that the NEXT group's rows are prefetched while this one is written;
        // they are other rows.
    }
    const XConst &c = inverse ? p.xw32->inv : p.xw32->fwd;
    const bool fpint = p.xw32->fpint;
#ifndef XW32_VARIANTS
#define XW32_VARIANTS 0x3F
#endif
    switch (p.variant) {
#if XW32_VARIANTS & 1
    case V_REFERENCE:  return launch_xv<V_REFERENCE>(p, inverse, out, a, count, c, st);
#endif
#if XW32_VARIANTS & 2
    case V_BARRETT:    return launch_xv<V_BARRETT>(p, inverse, out, a, count, c, st);
#endif
#if XW32_VARIANTS & 4
    case V_FP:
        if (!fpint) return launch_xv<V_FP>(p, inverse, out, a, count, c, st);
        return p.tw_bits == 16 ? launch_xv<V_FPI>(p, inverse, out, a, count, c, st) : launch_xv<V_FPG>(p, inverse, out, a, count, c, st);
#endif
#if XW32_VARIANTS & 8
    case V_AVX:
        // single-precision lanes for 16-bit tables with q <= 12289 (:1367-1402); the magic-number rounding needs q > 512
        if (p.tw_bits == 16 && p.rc.q <= 12289) {
            if (p.rc.q <= 512) return SCGPU_ERR_UNSUPPORTED;
            return fpint ? launch_xv<V_AVXFI>(p, inverse, out, a, count, c, st) : launch_xv<V_AVXF>(p, inverse, out, a, count, c, st);
        }
        if (!fpint) return launch_xv<V_AVX>(p, inverse, out, a, count, c, st);
        return p.tw_bits == 16 ? launch_xv<V_AVXI>(p, inverse, out, a, count, c, st) : launch_xv<V_AVXG>(p, inverse, out, a, count, c, st);
#endif
#if XW32_VARIANTS & 16
    case V_SOL7681:    return launch_xv<V_SOL7681>(p, inverse, out, a, count, c, st);
#endif
#if XW32_VARIANTS & 32
    case V_SOL8380417: return launch_xv<V_SOL8380417>(p, inverse, out, a, count, c, st);
#endif
    default:           return SCGPU_ERR_UNSUPPORTED;
    }
}

}  // namespace scgpu
