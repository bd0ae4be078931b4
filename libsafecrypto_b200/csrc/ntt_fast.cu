// ntt_fast.cu -- fused negacyclic products with canonical output.
//
//   polymul:  out = INTT(NTT(a) o NTT(b))          two operands in, one result out: 12 n bytes of HBM
//   mul_key:  out = INTT(NTT(t) o key)             key already in the reference's NTT domain
//   matvec:   t_i = INTT(sum_j A_ij o NTT(s_j))    module-LWE product (module_lwe.c:588-748)
//   each with an optional addend e (the *_add entry points): out = (product + e) mod q
//
// The result of these compositions is the canonical residue in [0, q) in the reference
// (inv_ntt_* ends with ntt32_flip_generic's conditional +q / -q, ntt.c:571-604), so the
// arithmetic inside is free (SURVEY.md 8a, representative contract rule 1).  What is used:
//
//  * merged-twiddle Cooley-Tukey forward / Gentleman-Sande inverse over psi = w[1] (the caller's
//    own 2n-th root): no separate pre/post twist, no bit-reversal pass.  Forward output index i
//    holds the reference's NTT-domain coefficient brv(i), which is how `key` / `A` are addressed.
//  * signed Montgomery products, R = 2^32: IMAD + 2 x IMAD.HI per twiddle multiply, the final
//    subtraction folded into the butterfly's 3-input adds; sums stay lazily reduced.
//  * n/8 threads per polynomial, 8 coefficients per thread: each pass does three radix-2 stages
//    in registers; between passes coefficients go through an XOR-swizzled shared-memory tile
//    (conflict-free for every pass's stride, checked in tests/test_layout.py); the polynomial never
//    leaves the SM between the first load and the final store.
//  * both operands of a product share the twiddle registers of a pass.
//  * arbitrary SINT32 inputs: the pass-through half of the first stage is range-compressed by
//    x - (x >> ceil(log2 q)) * q, everything else is bounded by the Montgomery products.
#include "scgpu_internal.h"
#include "fast_common.cuh"
#include "../../include/scgpu.h"

#include <atomic>
#include <cstdlib>
#include <vector>

namespace scgpu {

namespace {

using namespace fast;

__device__ __forceinline__ MontTw ld_tw(const MontTw *p)
{
    int2 v = __ldg(reinterpret_cast<const int2 *>(p));
    MontTw t; t.w = v.x; t.wq = v.y;
    return t;
}

// Twiddles of one pass for one thread: slot distance 4 -> 1 value, 2 -> 2 values, 1 -> 4 values.
struct PassTw { MontTw z4; MontTw z2[2]; MontTw z1[4]; };

template <int LOGN, int PASS>
__device__ __forceinline__ void load_pass_tw(PassTw &tw, const MontTw *zt, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    const int blk = tau / C::D;
    // stage with slot distance delta sits at s = S0 + (J - 1 - log2(delta)); table index 2^s + b
    if (C::J == 3) {
        tw.z4 = ld_tw(zt + (1 << C::S0) + blk);
    }
    if (C::J >= 2) {
        const int s = C::S0 + C::J - 2;
        tw.z2[0] = ld_tw(zt + (1 << s) + 2 * blk);
        tw.z2[1] = ld_tw(zt + (1 << s) + 2 * blk + 1);
    }
    {
        const int s = C::S0 + C::J - 1;
#pragma unroll
        for (int i = 0; i < 4; i++) tw.z1[i] = ld_tw(zt + (1 << s) + 4 * blk + i);
    }
}

__device__ __forceinline__ void ct_bfly(int32_t &lo, int32_t &hi, MontTw z, int32_t q)
{
    int32_t t = mont_mul(hi, z, q);
    hi = lo - t;
    lo = lo + t;
}
__device__ __forceinline__ void gs_bfly(int32_t &lo, int32_t &hi, MontTw z, int32_t q)
{
    int32_t d = lo - hi;
    lo = lo + hi;
    hi = mont_mul(d, z, q);
}

template <int J>
__device__ __forceinline__ void fwd_pass(int32_t (&x)[8], const PassTw &tw, int32_t q)
{
    if (J == 3) {
#pragma unroll
        for (int m = 0; m < 4; m++) ct_bfly(x[m], x[m + 4], tw.z4, q);
    }
    if (J >= 2) {
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) ct_bfly(x[m], x[m + 2], tw.z2[m >> 2], q);
    }
#pragma unroll
    for (int m = 0; m < 8; m += 2) ct_bfly(x[m], x[m + 1], tw.z1[m >> 1], q);
}

template <int J>
__device__ __forceinline__ void inv_pass(int32_t (&x)[8], const PassTw &tw, int32_t q)
{
#pragma unroll
    for (int m = 0; m < 8; m += 2) gs_bfly(x[m], x[m + 1], tw.z1[m >> 1], q);
    if (J >= 2) {
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) gs_bfly(x[m], x[m + 2], tw.z2[m >> 2], q);
    }
    if (J == 3) {
#pragma unroll
        for (int m = 0; m < 4; m++) gs_bfly(x[m], x[m + 4], tw.z4, q);
    }
}

struct FastConst {
    const MontTw *zf;
    const MontTw *zi;
    MontTw ninv, rsq, rone;
    int32_t q, qinv;
    int qbits;          // ceil(log2 q)
    int bigq;           // q * n >= 2^30: re-reduce between inverse passes
};

// ---- forward transform of one or two operands held in registers ---------------------------------
template <int LOGN, int PASS, int NOPS>
__device__ __forceinline__ void fwd_all(int32_t (&xa)[8], int32_t (&xb)[8], int32_t *ta, int32_t *tb,
                                        const FastConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    PassTw tw;
    load_pass_tw<LOGN, PASS>(tw, c.zf, tau);
    if (PASS > 0) {
        group_sync<LOGN>();
        tile_load<LOGN, PASS>(ta, xa, tau);
        if (NOPS == 2) tile_load<LOGN, PASS>(tb, xb, tau);
    }
    fwd_pass<C::J>(xa, tw, c.q);
    if (NOPS == 2) fwd_pass<C::J>(xb, tw, c.q);
    if constexpr (PASS + 1 < NumPasses<LOGN>::value) {
        tile_store<LOGN, PASS>(ta, xa, tau);
        if (NOPS == 2) tile_store<LOGN, PASS>(tb, xb, tau);
        fwd_all<LOGN, PASS + 1, NOPS>(xa, xb, ta, tb, c, tau);
    }
}

// ---- inverse transform, last pass first; ends with n^-1 scaling and canonical output -------------
template <int LOGN, int PASS>
__device__ __forceinline__ void inv_all(int32_t (&x)[8], int32_t *tile, const FastConst &c, int tau)
{
    using C = PassCfg<LOGN, PASS>;
    PassTw tw;
    load_pass_tw<LOGN, PASS>(tw, c.zi, tau);
    if (PASS + 1 < NumPasses<LOGN>::value) {
        group_sync<LOGN>();
        tile_load<LOGN, PASS>(tile, x, tau);
    }
    if constexpr (PASS == 0) {
        // last pass: stages 2, 1 then stage 0, whose twiddle already carries n^-1 on the difference
        // branch; the sum branch is scaled by n^-1 explicitly
#pragma unroll
        for (int m = 0; m < 8; m += 2) gs_bfly(x[m], x[m + 1], tw.z1[m >> 1], c.q);
#pragma unroll
        for (int m = 0; m < 8; m++) if ((m & 2) == 0) gs_bfly(x[m], x[m + 2], tw.z2[m >> 2], c.q);
#pragma unroll
        for (int m = 0; m < 4; m++) {
            int32_t s = x[m] + x[m + 4];
            int32_t d = x[m] - x[m + 4];
            x[m] = mont_mul(s, c.ninv, c.q);
            x[m + 4] = mont_mul(d, tw.z4, c.q);
        }
#pragma unroll
        for (int m = 0; m < 8; m++) x[m] += (x[m] >> 31) & c.q;
    } else {
        inv_pass<C::J>(x, tw, c.q);
        if (c.bigq) {
#pragma unroll
            for (int m = 0; m < 8; m++) x[m] = mont_mul(x[m], c.rone, c.q);
        }
        tile_store<LOGN, PASS>(tile, x, tau);
        inv_all<LOGN, PASS - 1>(x, tile, c, tau);
    }
}

template <int LOGN>
__device__ __forceinline__ void load_operand(int32_t (&x)[8], const int32_t *row, int tau, const FastConst &c)
{
    constexpr int D0 = PassCfg<LOGN, 0>::D;
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = __ldg(row + tau + m * D0);
    // pass-through half of stage 0: keep |x| < 2^31 - (log2 n + 1) q for any SINT32 input
#pragma unroll
    for (int m = 0; m < 4; m++) x[m] -= (x[m] >> c.qbits) * c.q;
}

enum { MODE_POLYMUL = 0, MODE_KEY16 = 1, MODE_KEY32 = 2 };

template <int LOGN, int MODE>
__global__ void __launch_bounds__(kCtaThreads)
k_polymul(int32_t *__restrict__ out, const int32_t *__restrict__ a, const void *__restrict__ bsrc,
          size_t b_stride, size_t count, FastConst c)
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
        load_operand<LOGN>(xa, a + prow * N, tau, c);
        if (MODE == MODE_POLYMUL) {
            load_operand<LOGN>(xb, static_cast<const int32_t *>(bsrc) + prow * b_stride, tau, c);
            fwd_all<LOGN, 0, 2>(xa, xb, ta, tb, c, tau);
            // pointwise: bring b into Montgomery form (also fully reduces it), then a * b
#pragma unroll
            for (int m = 0; m < 8; m++) {
                int32_t bm = mont_mul(xb[m], c.rsq, c.q);
                xa[m] = mont_mul2(xa[m], bm, c.qinv, c.q);
            }
        } else {
            fwd_all<LOGN, 0, 1>(xa, xb, ta, tb, c, tau);
            // key[j] is the reference's NTT-domain coefficient j (canonical); this thread's slot m of
            // the last pass holds coefficient brv(8 tau + m)
#pragma unroll
            for (int m = 0; m < 8; m++) {
                const int j = (int)(__brev((unsigned)(elem_index<PassCfg<LOGN, LAST>::D>(tau, m))) >> (32 - LOGN));
                int32_t kv = (MODE == MODE_KEY16)
                    ? (int32_t)__ldg(static_cast<const int16_t *>(bsrc) + prow * b_stride + j)
                    : __ldg(static_cast<const int32_t *>(bsrc) + prow * b_stride + j);
                int32_t km = mont_mul(kv, c.rsq, c.q);
                xa[m] = mont_mul2(xa[m], km, c.qinv, c.q);
            }
        }
        inv_all<LOGN, LAST>(xa, ta, c, tau);
        if (live) {
            int32_t *orow = out + poly * N;
#pragma unroll
            for (int m = 0; m < 8; m++) orow[tau + m * D0] = xa[m];
        }
        group_sync<LOGN>();
    }
}

// ---- module-LWE matrix-vector product --------------------------------------------------------------
// One instance per thread group: forward the l secret polynomials once (kept in a shared-memory
// stash in NTT domain), then for each of the k rows accumulate A_ij o s_j in registers, one
// inverse transform per row.  A is read exactly once, s once, t written once: 4n(k l + l + k) bytes.
// SHARED_A: one matrix for every instance (instance stride 0)
template <int LOGN, int MAXL, bool SHARED_A = false>
__global__ void __launch_bounds__(kCtaThreads)
k_matvec(int32_t *__restrict__ out, const int32_t *__restrict__ A, const int32_t *__restrict__ s,
         int k, int l, size_t count, FastConst c)
{
    constexpr int N = 1 << LOGN;
    constexpr int T = N / 8;
    constexpr int G = kCtaThreads / T;
    constexpr int D0 = PassCfg<LOGN, 0>::D;
    constexpr int LAST = NumPasses<LOGN>::value - 1;
    __shared__ __align__(16) int32_t tiles[G][N];
    __shared__ __align__(16) int32_t stash[G][MAXL][N];   // NTT(s_j), Montgomery form, thread-private slots
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
            load_operand<LOGN>(x, s + (irow * l + j) * N, tau, c);
            fwd_all<LOGN, 0, 1>(x, dummy, tile, tile, c, tau);
#pragma unroll
            for (int m = 0; m < 8; m++) stash[g][j][m * T + tau] = mont_mul(x[m], c.rsq, c.q);
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
                    acc[m] += mont_mul2(__ldg(arow + idx), stash[g][j][m * T + tau], c.qinv, c.q);
                }
            }
            inv_all<LOGN, LAST>(acc, tile, c, tau);
            if (live) {
                int32_t *orow = out + (inst * k + i) * N;
#pragma unroll
                for (int m = 0; m < 8; m++) orow[tau + m * D0] = acc[m];
            }
            group_sync<LOGN>();
        }
    }
}

int64_t powmod(int64_t b, int64_t e, int64_t q)
{
    __int128 r = 1, x = b % q;
    while (e > 0) { if (e & 1) r = (r * x) % q; x = (x * x) % q; e >>= 1; }
    return (int64_t)r;
}

MontTw make_tw(int64_t v, int64_t q, uint32_t qinv)
{
    // v in [0, q): Montgomery form v * 2^32 mod q, centred to (-q/2, q/2]
    int64_t m = (int64_t)(((__int128)v << 32) % q);
    if (m > q / 2) m -= q;
    MontTw t;
    t.w = (int32_t)m;
    t.wq = (int32_t)((uint32_t)(int32_t)m * qinv);
    return t;
}

}  // namespace

struct MontState {
    MontTw *zeta_fwd;    // [n]: index 2^s + b  -> psi^brv(.) * R
    MontTw *zeta_inv;    // [n]: inverses, last-stage entries pre-multiplied by n^-1
    FastConst c;
};

int build_fast_tables(NttPlanDev &p, const int32_t *w_host)
{
    const int n = p.n;
    const int64_t q = p.rc.q;
    if ((q & 1) == 0 || q < 3 || q >= (1ll << 30)) return SCGPU_OK;      // fused kernels unavailable
    // the caller's table must be powers of a 2n-th root of unity: w[1]^n == -1
    const int64_t psi = ((int64_t)w_host[1] % q + q) % q;
    if (powmod(psi, n, q) != q - 1) return SCGPU_OK;
    uint32_t qinv = 1;
    for (int i = 0; i < 5; i++) qinv *= 2u - (uint32_t)q * qinv;         // Newton: q^-1 mod 2^32
    const int64_t ninv = powmod(n, q - 2, q);
    std::vector<MontTw> zf(n), zi(n);
    zf[0] = make_tw(1, q, qinv); zi[0] = zf[0];
    for (int k = 1; k < n; k++) {
        int e = 0;
        for (int b = 0; b < p.logn; b++) e |= ((k >> b) & 1) << (p.logn - 1 - b);
        int64_t z = (((int64_t)w_host[e] % q) + q) % q;                  // psi^brv(k)
        int64_t zinv = (q - (((int64_t)w_host[n - e] % q) + q) % q) % q; // psi^-e = -psi^(n-e)
        if (k == 1) zinv = (int64_t)(((__int128)zinv * ninv) % q);
        zf[k] = make_tw(z, q, qinv);
        zi[k] = make_tw(zinv, q, qinv);
    }
    MontState *s = p.mont = new MontState();
    SCGPU_CUDA_CHECK(cudaMalloc(&s->zeta_fwd, sizeof(MontTw) * n));
    SCGPU_CUDA_CHECK(cudaMalloc(&s->zeta_inv, sizeof(MontTw) * n));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->zeta_fwd, zf.data(), sizeof(MontTw) * n, cudaMemcpyHostToDevice));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->zeta_inv, zi.data(), sizeof(MontTw) * n, cudaMemcpyHostToDevice));
    FastConst &c = s->c;
    c.zf = s->zeta_fwd; c.zi = s->zeta_inv;
    c.ninv = make_tw(ninv, q, qinv);
    c.rsq = make_tw((int64_t)(((__int128)1 << 32) % q), q, qinv);      // value R -> stored as R^2 mod q
    c.q = (int32_t)q; c.qinv = (int32_t)qinv;
    c.qbits = 0;
    while ((1ll << c.qbits) < q) c.qbits++;
    c.bigq = (q << p.logn) >= (1ll << 30);
    // R mod q in Montgomery form is R^2 mod q ... "multiply by one": mont(x, R) = x
    c.rone = make_tw(1, q, qinv);
    return SCGPU_OK;
}

void free_fast_tables(NttPlanDev &p)
{
    if (!p.mont) return;
    cudaFree(p.mont->zeta_fwd);
    cudaFree(p.mont->zeta_inv);
    delete p.mont;
    p.mont = nullptr;
}

// Arithmetic of the fused kernels: 0 = automatic (float-quotient where its bounds are proven -- the warp-local
// 32-coefficient schedule for polymul / key products -- else 32-bit Barrett, else Montgomery), 1 = Montgomery
// for every modulus, 2 = Barrett-32 where applicable, 3 = float-quotient with the 8-coefficient schedule,
// 4 = Shoup products on the warp-local schedule for every modulus they can serve.
// SCGPU_FAST_ARITH / SCGPU_FORCE_MONT=1 set the initial value; tests switch it to cover all three.
static std::atomic<int> g_arith{-1};       // read by every launch path, written by the setters: atomic, not locked
static int arith_mode()
{
    int m = g_arith.load(std::memory_order_relaxed);
    if (m < 0) {
        m = 0;
        if (getenv("SCGPU_FORCE_MONT") && atoi(getenv("SCGPU_FORCE_MONT")) != 0) m = 1;
        if (getenv("SCGPU_FAST_ARITH")) m = atoi(getenv("SCGPU_FAST_ARITH")) & 7;
        int expect = -1;
        if (!g_arith.compare_exchange_strong(expect, m)) m = expect;
    }
    return m;
}
int set_fast_arith(int mode)
{
    const int old = arith_mode();
    g_arith.store(mode & 7);
    return old;
}
int set_force_montgomery(int on)
{
    const int old = arith_mode() == 1 ? 1 : 0;
    g_arith.store(on ? 1 : 0);
    return old;
}

namespace {

enum Arith { AR_NONE, AR_MONT, AR_SQ, AR_FQ, AR_FQ32, AR_SH32 };
enum FusedOp { OP_PRODUCT, OP_MATVEC, OP_CANONICAL };       // OP_PRODUCT: two-operand and key products

// what the plan's arithmetics serve; *_lmax: largest l of their mat-vec (0: none)
struct Caps {
    bool mont, sq, fq, fq32, sh32;
    int fq32_lmax, sh32_lmax;
};

// The arithmetic that runs an operation (l: the mat-vec's inner dimension) under arithmetic mode m.  AR_NONE: none
// serves it.  The canonical transforms exist on the warp-local schedules only and follow mode 4 alone.
Arith choose_arith(int m, const Caps &cp, FusedOp op, int l)
{
    if (op == OP_CANONICAL) {
        if (cp.sh32 && (m == 4 || !cp.fq32)) return AR_SH32;
        return cp.fq32 ? AR_FQ32 : AR_NONE;
    }
    const bool mv = op == OP_MATVEC;
    const bool sh32 = cp.sh32 && (!mv || l <= cp.sh32_lmax);
    if (mv && l > 4) {
        // only the Shoup-policy kernels take l at run time (Dilithium k = 6, l = 5).  A modulus the float-quotient
        // mat-vec serves (the small moduli) stays at l <= 4 under every arithmetic, as scgpu.h promises, not only
        // under the automatic one
        return sh32 && (m == 0 || m == 4) && !(cp.fq32 && cp.fq32_lmax > 0) ? AR_SH32 : AR_NONE;
    }
    if (m == 4 && sh32) return AR_SH32;
    if (m == 0 && cp.fq32 && (!mv || l <= cp.fq32_lmax)) return AR_FQ32;
    if ((m == 0 || m == 3) && cp.fq) return AR_FQ;
    if (m != 1 && cp.sq) return AR_SQ;
    if (m == 0 && sh32) return AR_SH32;
    return cp.mont ? AR_MONT : AR_NONE;
}

Arith choose_arith(const NttPlanDev &p, FusedOp op, int l = 1)
{
    const Caps cp{p.mont != nullptr, p.sq != nullptr, p.fq != nullptr, p.fq32 != nullptr, p.sh32 != nullptr,
                  fq32_matvec_lmax(p), sh32_matvec_lmax(p)};
    return choose_arith(arith_mode(), cp, op, l);
}

int fused_unavailable(const NttPlanDev &p)
{
    set_error("fused kernels need an odd q < 2^30 and a table with w[1]^n == -1 (q=%d n=%d)", p.rc.q, p.n);
    return SCGPU_ERR_UNSUPPORTED;
}

// out = (prod + e) mod q for a canonical prod and any SINT32 e (64-bit sum: q + e may leave 32 bits).  out may be prod.
__global__ void k_add_canonical(int32_t *out, const int32_t *prod, const int32_t *e, size_t words, int32_t q)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < words; i += (size_t)gridDim.x * blockDim.x) {
        const int64_t v = ((int64_t)prod[i] + (int64_t)e[i]) % q;
        out[i] = (int32_t)(v < 0 ? v + q : v);
    }
}

// The addend on the arithmetics whose kernels have no epilogue for it (Montgomery, 32-bit Barrett, the 8-coefficient
// float-quotient schedule: cross-checks of the warp-local kernels, which add it in the product's own kernel):
// product(P) writes the sibling call's result, then one elementwise kernel adds e.  P is out, or a stream-ordered
// scratch of the call when out is e itself.
template <class F>
int add_after(const NttPlanDev &p, int32_t *out, const int32_t *e, size_t words, cudaStream_t st, F &&product)
{
    int32_t *P = out;
    if (out == e) SCGPU_CUDA_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&P), words * sizeof(int32_t), st));
    int r = product(P);
    if (r == SCGPU_OK) {
        const size_t cap = (size_t)(p.sm_count > 0 ? p.sm_count : 148) * 8;
        const size_t blocks = (words + 255) / 256;
        r = launch_kernel(k_add_canonical, (unsigned)(blocks < cap ? blocks : cap), 256, 0, st, out, P, e, words, p.rc.q);
    }
    if (P != out) {
        const cudaError_t fe = cudaFreeAsync(P, st);
        if (r == SCGPU_OK && fe != cudaSuccess) { set_error("cudaFreeAsync failed: %s", cudaGetErrorString(fe)); r = SCGPU_ERR_CUDA; }
    }
    return r;
}

}  // namespace

int launch_polymul(const NttPlanDev &p, int32_t *out, const int32_t *a, const int32_t *b,
                   size_t b_stride, size_t count, cudaStream_t st, const int32_t *e)
{
    if (count == 0) return SCGPU_OK;
    const Arith ar = choose_arith(p, OP_PRODUCT);
    if (e && ar != AR_SH32 && ar != AR_FQ32)
        return add_after(p, out, e, count * p.n, st, [&](int32_t *P) { return launch_polymul(p, P, a, b, b_stride, count, st); });
    switch (ar) {
    case AR_SH32: return launch_polymul_sh32(p, 0, out, a, b, b_stride, count, st, e);
    case AR_FQ32: return launch_polymul_fq32(p, 0, out, a, b, b_stride, count, st, e);
    case AR_FQ:   return launch_polymul_fq(p, 0, out, a, b, b_stride, count, st);
    case AR_SQ:   return launch_polymul_sq(p, 0, out, a, b, b_stride, count, st);
    case AR_MONT: break;
    default:      return fused_unavailable(p);
    }
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 4);      // 4 resident 256-thread CTAs per SM
    return with_int<8, 9, 10>(p.logn, [&](auto L) {
        return launch_kernel(k_polymul<L, MODE_POLYMUL>, grid, kCtaThreads, 0, st, out, a, b, b_stride, count, p.mont->c);
    });
}

// normalize_32(fwd_ntt(a)) / inv_ntt(a) through the warp-local kernels; SCGPU_ERR_UNSUPPORTED when neither
// arithmetic policy serves the modulus (the caller then composes the variant-exact kernels)
int launch_ntt_canonical(const NttPlanDev &p, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t st)
{
    if (count == 0) return SCGPU_OK;
    switch (choose_arith(p, OP_CANONICAL)) {
    case AR_SH32: return launch_ntt_sh32(p, inverse, out, a, count, st);
    case AR_FQ32: return launch_ntt_fq32(p, inverse, out, a, count, st);
    default:      return SCGPU_ERR_UNSUPPORTED;
    }
}

int launch_mul_key(const NttPlanDev &p, int32_t *out, const int32_t *t, const void *key,
                   int key_bits, size_t key_stride, size_t count, cudaStream_t st, const int32_t *e)
{
    if (count == 0) return SCGPU_OK;
    if (key_bits != 16 && key_bits != 32) { set_error("key_bits must be 16 or 32"); return SCGPU_ERR_ARG; }
    const int mode = key_bits == 16 ? MODE_KEY16 : MODE_KEY32;
    const Arith ar = choose_arith(p, OP_PRODUCT);
    if (e && ar != AR_SH32 && ar != AR_FQ32)
        return add_after(p, out, e, count * p.n, st,
                         [&](int32_t *P) { return launch_mul_key(p, P, t, key, key_bits, key_stride, count, st); });
    switch (ar) {
    case AR_SH32: return launch_polymul_sh32(p, mode, out, t, key, key_stride, count, st, e);
    case AR_FQ32: return launch_polymul_fq32(p, mode, out, t, key, key_stride, count, st, e);
    case AR_FQ:   return launch_polymul_fq(p, mode, out, t, key, key_stride, count, st);
    case AR_SQ:   return launch_polymul_sq(p, mode, out, t, key, key_stride, count, st);
    case AR_MONT: break;
    default:      return fused_unavailable(p);
    }
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 4);
    return with_int<8, 9, 10>(p.logn, [&](auto L) {
        return with_int<MODE_KEY16, MODE_KEY32>(mode, [&](auto M) {
            return launch_kernel(k_polymul<L, M>, grid, kCtaThreads, 0, st, out, t, key, key_stride, count, p.mont->c);
        });
    });
}

int launch_matvec(const NttPlanDev &p, int32_t *out, const int32_t *A, const int32_t *s,
                  int k, int l, size_t count, cudaStream_t st, bool shared, const int32_t *e)
{
    if (count == 0) return SCGPU_OK;
    if (!p.mont) return fused_unavailable(p);
    if (k < 1 || l < 1 || l > 8) { set_error("matvec supports 1 <= l <= 8 (got k=%d l=%d)", k, l); return SCGPU_ERR_ARG; }
    if (p.logn != 8) { set_error("matvec is instantiated for n = 256 (Kyber / Dilithium); got n=%d", p.n); return SCGPU_ERR_UNSUPPORTED; }
    const Arith ar = choose_arith(p, OP_MATVEC, l);
    if (e && ar != AR_SH32 && ar != AR_FQ32)
        return add_after(p, out, e, count * (size_t)k * p.n, st,
                         [&](int32_t *P) { return launch_matvec(p, P, A, s, k, l, count, st, shared); });
    switch (ar) {
    case AR_SH32: return launch_matvec_sh32(p, out, A, s, k, l, count, st, shared, e);
    case AR_FQ32: return launch_matvec_fq32(p, out, A, s, k, l, count, st, shared, e);
    case AR_FQ:   return launch_matvec_fq(p, out, A, s, k, l, count, st, shared);
    case AR_SQ:   return launch_matvec_sq(p, out, A, s, k, l, count, st, shared);
    case AR_MONT: break;
    default:      set_error("matvec l > 4 not instantiated for this modulus"); return SCGPU_ERR_UNSUPPORTED;
    }
    const unsigned grid = cta_grid(p.sm_count, p.n, count, 4);
    if (shared) return launch_kernel(k_matvec<8, 4, true>, grid, kCtaThreads, 0, st, out, A, s, k, l, count, p.mont->c);
    return launch_kernel(k_matvec<8, 4>, grid, kCtaThreads, 0, st, out, A, s, k, l, count, p.mont->c);
}

}  // namespace scgpu
