// ntt_fast_sq.cu -- fused negacyclic products for SMALL moduli (q = 7681, 12289, ...): all modular
// products stay in 32 bits and are reduced with a round-to-nearest 32-bit Barrett step.
//
// Why a second arithmetic: on B200 the fma pipe issues IMAD at 64 lanes/clk/SM but IMAD.HI at 32
// (measured, profiles/int_peaks_r01.txt).  A Montgomery product (ntt_fast.cu) needs 2 x IMAD.HI + IMAD = 5
// fma slots; when |x * w| < 2^31 the product itself is one IMAD and
//       t = p - hi32(p * M + 2^31) * q ,   M = floor(2^32 / q)          (|t| < q)
// costs IMAD + IMAD.HI + IMAD = 4 slots, needs one 32-bit word per twiddle instead of two, and leaves no
// high-word subtraction for ptxas to fold into 64-bit accumulators (which cost 20 % of the issue slots in
// MOVs in the Montgomery kernel, profiles/polymul_r01a_mix.txt).
//
// Values are lazily reduced; the host proves at plan creation (sq_analyse) by interval propagation over
// exactly this kernel's dataflow that every product stays below 2^31, choosing how many cheap range
// compressions  x -= (x >> ceil(log2 q)) * q  to apply before the pointwise product and at the entry of each
// inverse pass.  If no schedule exists for (q, n) the plan falls back to the Montgomery kernels.
//
// Arbitrary SINT32 inputs: a warp votes on "any |x| > 4q in my 8 coefficients"; only then are the inputs
// Barrett-reduced first, so in-range operands (what every scheme passes) pay two ALU ops per coefficient.
#include "scgpu_internal.h"
#include "fast_common.cuh"
#include "../../include/scgpu.h"

#include <vector>

namespace scgpu {

using namespace fast;

namespace {

struct SqConst {
    const int32_t *zf;      // [n] psi^brv(k), centred
    const int32_t *zi;      // [n] inverses, entry 1 pre-multiplied by n^-1
    int32_t q, nq, M, ninv, x0; // nq = -q; M = floor(2^32/q); x0 = input magnitude the bounds were proven for
    int qbits;
    int r_pw;               // compress rounds before the pointwise product
    int r_inv[4];           // compress rounds at the entry of inverse pass p
};

// round-to-nearest Barrett on a 32-bit value: |result| < q for any |p| < 2^31
__device__ __forceinline__ int32_t bred(int32_t p, const SqConst &c)
{
    int32_t qe = (int32_t)(((int64_t)p * (int64_t)c.M + 0x80000000ll) >> 32);
    return qe * c.nq + p;           // one IMAD: no separate negation
}
__device__ __forceinline__ int32_t bmul(int32_t x, int32_t w, const SqConst &c) { return bred(x * w, c); }

__device__ __forceinline__ int32_t compress(int32_t x, int rounds, const SqConst &c)
{
    // rounds is a plan constant in 0..3 (uniform branches; a counted loop makes nvcc unroll by 8)
    if (rounds > 0) x = (x >> c.qbits) * c.nq + x;
    if (rounds > 1) x = (x >> c.qbits) * c.nq + x;
    if (rounds > 2) x = (x >> c.qbits) * c.nq + x;
    return x;
}

struct SqTw { int32_t z4; int32_t z2[2]; int32_t z1[4]; };

template <int LOGN, int PASS>
__device__ __forceinline__ void sq_load_tw(SqTw &tw, const int32_t *zt, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    const int blk = tau / C::D;
    if (C::J == 3) tw.z4 = __ldg(zt + (1 << C::S0) + blk);
    if (C::J >= 2) {
        const int s = C::S0 + C::J - 2;
        const int2 v = __ldg(reinterpret_cast<const int2 *>(zt + (1 << s) + 2 * blk));
        tw.z2[0] = v.x; tw.z2[1] = v.y;
    }
    {
        const int s = C::S0 + C::J - 1;
        const int4 v = __ldg(reinterpret_cast<const int4 *>(zt + (1 << s) + 4 * blk));
        tw.z1[0] = v.x; tw.z1[1] = v.y; tw.z1[2] = v.z; tw.z1[3] = v.w;
    }
}

__device__ __forceinline__ void sq_ct(int32_t &lo, int32_t &hi, int32_t z, const SqConst &c)
{
    int32_t t = bmul(hi, z, c);
    hi = lo - t;
    lo = lo + t;
}
__device__ __forceinline__ void sq_gs(int32_t &lo, int32_t &hi, int32_t z, const SqConst &c)
{
    int32_t d = lo - hi;
    lo = lo + hi;
    hi = bmul(d, z, c);
}

template <int J>
__device__ __forceinline__ void sq_fwd_pass(int32_t (&x)[8], const SqTw &tw, const SqConst &c)
{
    if (J == 3) {
#pragma unroll
        for (int m = 0; m < 4; m++) sq_ct(x[m], x[m + 4], tw.z4, c);
    }
    if (J >= 2) {
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) sq_ct(x[m], x[m + 2], tw.z2[m >> 2], c);
    }
#pragma unroll
    for (int m = 0; m < 8; m += 2) sq_ct(x[m], x[m + 1], tw.z1[m >> 1], c);
}

template <int LOGN, int PASS, int NOPS>
__device__ __forceinline__ void sq_fwd_all(int32_t (&xa)[8], int32_t (&xb)[8], int32_t *ta, int32_t *tb,
                                           const SqConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    SqTw tw;
    sq_load_tw<LOGN, PASS>(tw, c.zf, tau);
    if (PASS > 0) {
        group_sync<LOGN>();
        tile_load<LOGN, PASS>(ta, xa, tau);
        if (NOPS == 2) tile_load<LOGN, PASS>(tb, xb, tau);
    }
    sq_fwd_pass<C::J>(xa, tw, c);
    if (NOPS == 2) sq_fwd_pass<C::J>(xb, tw, c);
    if constexpr (PASS + 1 < NumPasses<LOGN>::value) {
        tile_store<LOGN, PASS>(ta, xa, tau);
        if (NOPS == 2) tile_store<LOGN, PASS>(tb, xb, tau);
        sq_fwd_all<LOGN, PASS + 1, NOPS>(xa, xb, ta, tb, c, tau);
    }
}

template <int LOGN, int PASS>
__device__ __forceinline__ void sq_inv_all(int32_t (&x)[8], int32_t *tile, const SqConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    SqTw tw;
    sq_load_tw<LOGN, PASS>(tw, c.zi, tau);
    if (PASS + 1 < NumPasses<LOGN>::value) {
        group_sync<LOGN>();
        tile_load<LOGN, PASS>(tile, x, tau);
    }
    if (c.r_inv[PASS]) {
#pragma unroll
        for (int m = 0; m < 8; m++) x[m] = compress(x[m], c.r_inv[PASS], c);
    }
#pragma unroll
    for (int m = 0; m < 8; m += 2) sq_gs(x[m], x[m + 1], tw.z1[m >> 1], c);
    if (C::J >= 2) {
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) sq_gs(x[m], x[m + 2], tw.z2[m >> 2], c);
    }
    if constexpr (PASS == 0) {
        // stage 0: both branches are multiplied (n^-1 on the sum, n^-1 * zeta^-1 on the difference),
        // then the canonical representative
#pragma unroll
        for (int m = 0; m < 4; m++) {
            int32_t s = x[m] + x[m + 4];
            int32_t d = x[m] - x[m + 4];
            x[m] = bmul(s, c.ninv, c);
            x[m + 4] = bmul(d, tw.z4, c);
        }
#pragma unroll
        for (int m = 0; m < 8; m++) x[m] += (x[m] >> 31) & c.q;
    } else {
        if (C::J == 3) {
#pragma unroll
            for (int m = 0; m < 4; m++) sq_gs(x[m], x[m + 4], tw.z4, c);
        }
        tile_store<LOGN, PASS>(tile, x, tau);
        sq_inv_all<LOGN, PASS - 1>(x, tile, c, tau);
    }
}

template <int LOGN>
__device__ __forceinline__ void sq_load_operand(int32_t (&x)[8], const int32_t *row, int tau, const SqConst &c)
{
    constexpr int D0 = PassCfg<LOGN, 0>::D;
    bool wide = false;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        x[m] = __ldg(row + tau + m * D0);
        wide |= ((uint32_t)x[m] + (uint32_t)c.x0) > (uint32_t)(2 * c.x0);
    }
    if (__any_sync(0xFFFFFFFFu, wide)) {
#pragma unroll
        for (int m = 0; m < 8; m++) x[m] = bred(x[m], c);
    }
}

enum { SQ_POLYMUL = 0, SQ_KEY16 = 1, SQ_KEY32 = 2 };

template <int LOGN, int MODE>
__global__ void __launch_bounds__(kCtaThreads, 4)
k_polymul_sq(int32_t *__restrict__ out, const int32_t *__restrict__ a, const void *__restrict__ bsrc,
             size_t b_stride, size_t count, SqConst c)
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
        int32_t xa[8], xb[8];
        sq_load_operand<LOGN>(xa, a + prow * N, tau, c);
        if (MODE == SQ_POLYMUL) {
            sq_load_operand<LOGN>(xb, static_cast<const int32_t *>(bsrc) + prow * b_stride, tau, c);
            sq_fwd_all<LOGN, 0, 2>(xa, xb, ta, tb, c, tau);
#pragma unroll
            for (int m = 0; m < 8; m++)
                xa[m] = bmul(compress(xa[m], c.r_pw, c), compress(xb[m], c.r_pw, c), c);
        } else {
            sq_fwd_all<LOGN, 0, 1>(xa, xb, ta, tb, c, tau);
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int j = (int)(__brev((unsigned)(elem_index<PassCfg<LOGN, LAST>::D>(tau, m))) >> (32 - LOGN));
                int32_t kv;
                if (MODE == SQ_KEY16) kv = (int32_t)__ldg(static_cast<const int16_t *>(bsrc) + prow * b_stride + j);
                else                  kv = bred(__ldg(static_cast<const int32_t *>(bsrc) + prow * b_stride + j), c);
                xa[m] = bmul(compress(xa[m], c.r_pw, c), kv, c);
            }
        }
        sq_inv_all<LOGN, LAST>(xa, ta, c, tau);
        if (live) {
            int32_t *orow = out + poly * N;
#pragma unroll
            for (int m = 0; m < 8; m++) orow[tau + m * D0] = xa[m];
        }
        group_sync<LOGN>();
    }
}

// module-LWE matrix-vector product, same structure as k_matvec in ntt_fast.cu
// SHARED_A: one matrix for every instance (instance stride 0)
template <int LOGN, int MAXL, bool SHARED_A = false>
__global__ void __launch_bounds__(kCtaThreads)
k_matvec_sq(int32_t *__restrict__ out, const int32_t *__restrict__ A, const int32_t *__restrict__ s,
            int k, int l, size_t count, SqConst c)
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
        int32_t dummy[8];
        for (int j = 0; j < l; j++) {
            int32_t x[8];
            sq_load_operand<LOGN>(x, s + (irow * l + j) * N, tau, c);
            sq_fwd_all<LOGN, 0, 1>(x, dummy, tile, tile, c, tau);
#pragma unroll
            for (int m = 0; m < 8; m++) stash[g][j][m * T + tau] = bred(x[m], c);      // |.| < q
            group_sync<LOGN>();
        }
        for (int i = 0; i < k; i++) {
            int32_t acc[8];
#pragma unroll
            for (int m = 0; m < 8; m++) acc[m] = 0;
            for (int j = 0; j < l; j++) {
                const int32_t *arow = A + (((SHARED_A ? (size_t)0 : irow * k) + i) * l + j) * N;
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    const int idx = (int)(__brev((unsigned)(elem_index<PassCfg<LOGN, LAST>::D>(tau, m))) >> (32 - LOGN));
                    // A is canonical in the reference (sampled in [0, q)); reduce anyway so any SINT32 is exact
                    acc[m] += bmul(bred(__ldg(arow + idx), c), stash[g][j][m * T + tau], c);
                }
            }
            sq_inv_all<LOGN, LAST>(acc, tile, c, tau);
            if (live) {
                int32_t *orow = out + (inst * k + i) * N;
#pragma unroll
                for (int m = 0; m < 8; m++) orow[tau + m * D0] = acc[m];
            }
            group_sync<LOGN>();
        }
    }
}

int64_t powmod64(int64_t b, int64_t e, int64_t q)
{
    __int128 r = 1, x = b % q;
    while (e > 0) { if (e & 1) r = (r * x) % q; x = (x * x) % q; e >>= 1; }
    return (int64_t)r;
}

int32_t centre(int64_t v, int64_t q) { return (int32_t)(v > q / 2 ? v - q : v); }

}  // namespace

// Interval propagation over the kernel's dataflow.  All magnitudes are upper bounds on |value|.
// Returns true and fills sc's compress schedule when every 32-bit product is provably below 2^31.
static bool sq_analyse(const NttPlanDev &p, SqConst &sc, int max_accumulate)
{
    const double q = p.rc.q, lim = 2147483647.0;
    const double wmax = (double)(p.rc.q / 2);           // centred twiddles
    const int L = sc.qbits;
    const double f = 1.0 - q / (double)(1ll << L);      // compress: |x'| <= f |x| + q
    auto comp = [&](double b, int rounds) { for (int r = 0; r < rounds; r++) b = f * b + q; return b; };
    const double t = q;                                 // |bred(.)| < q for any 32-bit argument
    // forward: additive growth from the proven input magnitude
    double bf = sc.x0;
    for (int s = 0; s < p.logn; s++) {
        if (bf * wmax >= lim) return false;
        bf += t;
    }
    // pointwise: both operands compressed r_pw times (key products: one operand is < 2^15 or < q)
    int r_pw = -1;
    for (int r = 0; r <= 3; r++) {
        double c = comp(bf, r);
        if (c * c < lim && c * (q > 32768.0 ? q : 32768.0) < lim) { r_pw = r; break; }
    }
    if (r_pw < 0) return false;
    sc.r_pw = r_pw;
    // inverse passes, last pass of the schedule first; matvec accumulates up to max_accumulate products
    const int npass = (p.logn + 2) / 3;
    double bin = t * max_accumulate;
    for (int pass = npass - 1; pass >= 0; pass--) {
        const int J = (p.logn - 3 * pass) >= 3 ? 3 : (p.logn - 3 * pass);
        int chosen = -1;
        double bout = 0;
        for (int r = 0; r <= 3 && chosen < 0; r++) {
            double b[8];
            for (int m = 0; m < 8; m++) b[m] = comp(bin, r);
            bool ok = true;
            for (int st = 0; st < J && ok; st++) {
                const int delta = 1 << st;
                const bool last = (pass == 0 && st == J - 1);
                for (int m = 0; m < 8 && ok; m++) {
                    if (m & delta) continue;
                    double d = b[m] + b[m + delta];
                    if (d * wmax >= lim) ok = false;
                    b[m] = last ? t : d;
                    b[m + delta] = t;
                }
            }
            if (ok) {
                chosen = r;
                for (int m = 0; m < 8; m++) bout = b[m] > bout ? b[m] : bout;
            }
        }
        if (chosen < 0) return false;
        sc.r_inv[pass] = chosen;
        bin = bout;
    }
    return true;
}

struct SqState {
    int32_t *zf, *zi;
    SqConst prod, mv;       // mv: compress schedule for up to 4 accumulated products
};

int build_sq_tables(NttPlanDev &p, const int32_t *w_host)
{
    const int n = p.n;
    const int64_t q = p.rc.q;
    if ((q & 1) == 0 || q < 257 || q >= (1 << 20) || p.logn < 8 || p.logn > 10) return SCGPU_OK;
    const int64_t psi = (((int64_t)w_host[1] % q) + q) % q;
    if (powmod64(psi, n, q) != q - 1) return SCGPU_OK;
    SqConst c{};
    c.q = (int32_t)q; c.nq = (int32_t)-q;
    while ((1ll << c.qbits) < q) c.qbits++;
    c.M = (int32_t)(uint32_t)((1ull << 32) / (uint64_t)q);
    c.x0 = (int32_t)(4 * q);
    SqConst mv = c;
    // products can exceed 32 bits for this (q, n): the Montgomery kernels serve it
    if (!sq_analyse(p, c, 1) || !sq_analyse(p, mv, 4)) return SCGPU_OK;
    const int64_t ninv = powmod64(n, q - 2, q);
    std::vector<int32_t> zf(n), zi(n);
    zf[0] = zi[0] = 1;
    for (int k = 1; k < n; k++) {
        int e = 0;
        for (int b = 0; b < p.logn; b++) e |= ((k >> b) & 1) << (p.logn - 1 - b);
        int64_t z = (((int64_t)w_host[e] % q) + q) % q;
        int64_t zinv = (q - (((int64_t)w_host[n - e] % q) + q) % q) % q;
        if (k == 1) zinv = (int64_t)(((__int128)zinv * ninv) % q);
        zf[k] = centre(z, q);
        zi[k] = centre(zinv, q);
    }
    SqState *s = p.sq = new SqState();
    SCGPU_CUDA_CHECK(cudaMalloc(&s->zf, sizeof(int32_t) * n));
    SCGPU_CUDA_CHECK(cudaMalloc(&s->zi, sizeof(int32_t) * n));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->zf, zf.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->zi, zi.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    c.zf = mv.zf = s->zf;
    c.zi = mv.zi = s->zi;
    c.ninv = mv.ninv = centre(ninv, q);
    s->prod = c;
    s->mv = mv;
    return SCGPU_OK;
}

void free_sq_tables(NttPlanDev &p)
{
    if (!p.sq) return;
    cudaFree(p.sq->zf);
    cudaFree(p.sq->zi);
    delete p.sq;
    p.sq = nullptr;
}

int launch_polymul_sq(const NttPlanDev &p, int mode, int32_t *out, const int32_t *a, const void *b,
                      size_t b_stride, size_t count, cudaStream_t st)
{
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 4);
    return with_int<8, 9, 10>(p.logn, [&](auto L) {
        return with_int<SQ_POLYMUL, SQ_KEY16, SQ_KEY32>(mode, [&](auto M) {
            return launch_kernel(k_polymul_sq<L, M>, grid, kCtaThreads, 0, st, out, a, b, b_stride, count, p.sq->prod);
        });
    });
}

int launch_matvec_sq(const NttPlanDev &p, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                     size_t count, cudaStream_t st, bool shared)
{
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 2);
    if (shared) return launch_kernel(k_matvec_sq<8, 4, true>, grid, kCtaThreads, 0, st, out, A, s, k, l, count, p.sq->mv);
    return launch_kernel(k_matvec_sq<8, 4>, grid, kCtaThreads, 0, st, out, A, s, k, l, count, p.sq->mv);
}

}  // namespace scgpu
