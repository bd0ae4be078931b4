// ntt_fast_fq32.cu -- fused negacyclic product, float-quotient arithmetic (fq_arith.cuh) on the WARP-LOCAL schedule
// of warp32.cuh (which is generic in the arithmetic; this file supplies the policy ArFq and the host set-up):
// 32 coefficients per thread, n/32 threads per polynomial (8 / 16 / 32 lanes of ONE warp for n = 256 / 512 /
// 1024), so a whole product needs one shared-memory exchange per transform and only __syncwarp():
//
//   pass 0   stages 0..4   thread tau holds elements tau + (n/32) m, m = 0..31.  The 31 twiddles of these
//                          stages are the same for every thread: they live in the kernel's constant bank, or, for
//                          the reference's (12289, 512) table, in the instructions themselves (ArFqImm).
//   pass 1   stages 5..    thread tau holds the 32 contiguous elements 32 tau .. 32 tau + 31, i.e. 32 / SUB
//                          independent sub-chunks of SUB = n/32 elements; both operands of a sub-chunk are
//                          transformed together (shared twiddles), multiplied pointwise and taken back through
//                          the inverse stages before the next sub-chunk is touched.
//
// Against the 8-coefficient schedule of ntt_fast_fq.cu (per product, n = 512): 2 exchanges instead of 6
// (96 instead of 192 shared-memory wavefronts), no named barriers, address arithmetic amortised over 4x more
// butterflies, 16 independent butterflies per stage per thread.  The tile is padded (4 words per 32 elements)
// so that both the strided 32-bit accesses of pass 0 and the 128-bit accesses of pass 1 are conflict-free and
// every address is  thread base + compile-time offset.  Pass-1 twiddles are stored thread-major per stage
// (fq32_slot) so that a warp's 128-bit twiddle loads are contiguous.
#include "warp32.cuh"
#include "fq_host.h"

#include <algorithm>
#include <cstring>
#include <type_traits>
#include <utility>
#include <vector>

namespace scgpu {

namespace {

using fq::Tw;
using fq::kBias;
using w32::u32;

// Arithmetic policy: float-quotient products (fq_arith.cuh); coefficients travel biased by kBias.
struct ArFq {
    typedef Tw E;
    struct K { int32_t nq, q, pwk; float invq; int32_t pwb; float two23; };   // two23 = 2^23: ArFqImm's FFMA addend
    static constexpr bool STASH16 = true;          // mat-vec may keep the transformed vectors as int16
    static constexpr bool BASEMUL = true;          // two-operand products stop two stages early (fq::basemul4)
    static constexpr int WORDS = 4;
    static constexpr bool PASS0_IMM = false;
    template <int L, int M, bool BM> static constexpr bool serves() { return true; }
    static __device__ __forceinline__ u32 enc(int32_t x) { return (u32)x + (u32)kBias; }
    static __device__ __forceinline__ int32_t dec(u32 x) { return (int32_t)(x - (u32)kBias); }
    static __device__ __forceinline__ u32 zero() { return (u32)kBias; }
    // w and wq are used as constant-bank operands, k and c come as one 64-bit constant load
    static __device__ __forceinline__ E cb(const E &e)
    {
        const int2 kc = *reinterpret_cast<const int2 *>(&e.k);
        E t;
        t.w = e.w; t.wq = e.wq; t.k = kc.x; t.c = __int_as_float(kc.y);
        return t;
    }
    static __device__ __forceinline__ E mk(const int32_t (&w)[4])
    {
        return E{w[0], __int_as_float(w[1]), w[2], __int_as_float(w[3])};
    }
    static __device__ __forceinline__ void ct(u32 &lo, u32 &hi, const E &z, const K &k)
    {
        const u32 t = (u32)fq::mul((int32_t)hi, z, k.nq);
        hi = lo - t;
        lo = lo + t;
    }
    static __device__ __forceinline__ void ct0(u32 &lo, u32 &hi, const E &z, const K &k)
    {
        const u32 t = (u32)fq::mul((int32_t)hi, z, k.nq);
#ifdef __CUDA_ARCH__
        // two opaque copies of kBias: written with the literal, the compiler shares (lo + kBias) between the two
        // results (3 adds per pair); with distinct values each result is one 3-input IADD3
        u32 kb1, kb2;
        asm("mov.u32 %0, 0x4B400000;" : "=r"(kb1));
        asm("mov.u32 %0, 1262485504;" : "=r"(kb2));
        hi = lo - t + kb1;
        lo = lo + t + kb2;
#else
        hi = lo - t + (u32)kBias;
        lo = lo + t + (u32)kBias;
#endif
    }
    // both results UNBIASED (the stage in front of the base multiplication): the bias leaves inside the 3-input adds
    static __device__ __forceinline__ void ct_unb(u32 &lo, u32 &hi, const E &z, const K &k)
    {
        const u32 t = (u32)fq::mul((int32_t)hi, z, k.nq);
#ifdef __CUDA_ARCH__
        u32 kb1, kb2;                                    // opaque copies, see ct0
        asm("mov.u32 %0, 0x4B400000;" : "=r"(kb1));
        asm("mov.u32 %0, 1262485504;" : "=r"(kb2));
        hi = lo - t - kb1;
        lo = lo + t - kb2;
#else
        hi = lo - t - (u32)kBias;
        lo = lo + t - (u32)kBias;
#endif
    }
    // xa[0..3] (unbiased) <- xa * xb modulo X^4 - zeta, biased
    static __device__ __forceinline__ void bm4(u32 *xa, const u32 *xb, int32_t zw, int32_t zwq, const K &k)
    {
        int32_t a[4], b[4], c[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { a[i] = (int32_t)xa[i]; b[i] = (int32_t)xb[i]; }
        fq::basemul4(c, a, b, zw, __int_as_float(zwq), k.invq, k.pwk, k.pwb, k.nq);
#pragma unroll
        for (int i = 0; i < 4; i++) xa[i] = (u32)c[i];
    }
    // xa[0..3] (unbiased) <- xa * key modulo X^4 - zeta, biased; the four vectors are one block of the residue table
    static __device__ __forceinline__ void bmk4(u32 *xa, const int4 &vb, const int4 &vbf, const int4 &vz, const int4 &vzf, const K &k)
    {
        int32_t a[4], c[4];
#pragma unroll
        for (int i = 0; i < 4; i++) a[i] = (int32_t)xa[i];
        const int32_t b[4] = {vb.x, vb.y, vb.z, vb.w}, zb[4] = {vz.x, vz.y, vz.z, vz.w};
        const float bf[4] = {__int_as_float(vbf.x), __int_as_float(vbf.y), __int_as_float(vbf.z), __int_as_float(vbf.w)};
        const float zbf[4] = {__int_as_float(vzf.x), __int_as_float(vzf.y), __int_as_float(vzf.z), __int_as_float(vzf.w)};
        fq::basemul4_key(c, a, b, bf, zb, zbf, k.invq, k.pwb, k.nq);
#pragma unroll
        for (int i = 0; i < 4; i++) xa[i] = (u32)c[i];
    }
    static __device__ __forceinline__ void gs(u32 &lo, u32 &hi, const E &z, const K &k)
    {
        const u32 d = lo - hi + (u32)kBias;
        lo = lo + hi - (u32)kBias;
        hi = (u32)fq::mul((int32_t)d, z, k.nq);          // z.k carries the bias of the result
    }
    // both products are unbiased and proven to lie in (-q, q): one conditional +q gives the canonical residue
    static __device__ __forceinline__ void fin(u32 &lo, u32 &hi, const E &ninv, const E &z, const K &k)
    {
        const u32 s = lo + hi - (u32)kBias;
        const u32 d = lo - hi + (u32)kBias;
        const u32 ys = (u32)fq::mul((int32_t)s, ninv, k.nq);
        const u32 yd = (u32)fq::mul((int32_t)d, z, k.nq);
        lo = min(ys, ys + (u32)k.q);
        hi = min(yd, yd + (u32)k.q);
    }
    static __device__ __forceinline__ u32 red(u32 x, const E &one, const K &k) { return (u32)fq::mul((int32_t)x, one, k.nq); }
    static __device__ __forceinline__ u32 pw(u32 a, u32 b, const K &k)
    {
        return (u32)fq::mul_var(dec(a), dec(b), k.invq, k.pwk, k.nq) + (u32)kBias;
    }
    static __device__ __forceinline__ u32 pwraw(u32 a, int32_t kv, const K &k)
    {
        return (u32)fq::mul_var(dec(a), kv, k.invq, k.pwk, k.nq) + (u32)kBias;
    }
    // mat-vec accumulator: the l products of an output coefficient share ONE quotient.  p = sum of the low
    // products (wrap-around), f = the same sum in floats (each product below 2^32, l <= 8: the float error is a
    // few thousand, i.e. a fraction of q in the quotient); acc_fin = p - rint(f / q) q, biased.
    struct Acc { u32 p; float f; };
    static __device__ __forceinline__ Acc acc_zero() { return Acc{0u, 0.0f}; }
    static __device__ __forceinline__ void acc_add(Acc &a, int32_t av, int32_t sv, const K &)
    {
        a.p = (u32)fq::mad(av, sv, (int32_t)a.p);
        a.f = __fmaf_rn(__int2float_rn(av), __int2float_rn(sv), a.f);
    }
    // the same from an exact 32-bit sum (no wrap-around): one conversion, one quotient
    static __device__ __forceinline__ u32 acc_fin_int(int32_t p, const K &k)
    {
        const float f = __fmaf_rn(__int2float_rn(p), k.invq, fq::kBiasF);
        return (u32)fq::mad(fq::as_i(f), k.nq, (int32_t)((u32)p + (u32)k.pwk)) + (u32)kBias;
    }
    static __device__ __forceinline__ u32 acc_fin(const Acc &a, const K &k)
    {
        const float f = __fmaf_rn(a.f, k.invq, fq::kBiasF);
        return (u32)fq::mad(fq::as_i(f), k.nq, (int32_t)(a.p + (u32)k.pwk)) + (u32)kBias;
    }
};

typedef w32::W32Const<ArFq> FqConst32;

// ---- pass 0 of the reference's (q, n) = (12289, 512) table, compiled in ------------------------------------------
// The reference's ntt_table_gen table is w[e] = psi^e, psi the smallest m >= 2 with m^n = -1 (mod q).  From it
// build_tables / build_bm_tables derive the pass-0 entries zf[k] = psi^brv(k) and zi[k] = -psi^(n - brv(k)), and for the
// last stage of the base-multiplication schedule (n/4)^-1 and zi[1] (n/4)^-1.  The same formulas, evaluated by the
// compiler, make every pass-0 entry of the fused product an instruction immediate (fq_arith.cuh: make_imm): no constant
// loads, no registers.  build_fq32_tables selects this kernel only when the plan's own entries equal these.
namespace p0 {
constexpr int64_t kQ = 12289;
constexpr int kLogN = 9, kN = 1 << kLogN;
constexpr int64_t pow_c(int64_t b, int64_t e)
{
    int64_t r = 1;
    for (b %= kQ; e > 0; e >>= 1, b = b * b % kQ)
        if (e & 1) r = r * b % kQ;
    return r;
}
constexpr int64_t first_root()
{
    for (int64_t m = 2; m < kQ - 1; m++)
        if (pow_c(m, kN) == kQ - 1) return m;
    return 0;
}
constexpr int64_t kPsi = first_root();
constexpr int brv(int k)
{
    int e = 0;
    for (int b = 0; b < kLogN; b++) e |= ((k >> b) & 1) << (kLogN - 1 - b);
    return e;
}
constexpr int64_t fwd(int k) { return pow_c(kPsi, brv(k)); }                       // zf[k].w
constexpr int64_t inv(int k) { return (kQ - pow_c(kPsi, kN - brv(k))) % kQ; }     // zi[k].w, k >= 2
constexpr int64_t ninv() { return pow_c(kN / 4, kQ - 2); }                         // (n/4)^-1
constexpr int64_t inv1() { return inv(1) * ninv() % kQ; }                          // zi[1] (n/4)^-1
static_assert(kPsi != 0 && pow_c(kPsi, 2 * kN) == 1, "no 2n-th root of unity");

template <int... I, class F>
__device__ __forceinline__ void static_for_(std::integer_sequence<int, I...>, F &&f) { (f(std::integral_constant<int, I>{}), ...); }
template <int N, class F>
__device__ __forceinline__ void static_for(F &&f) { static_for_(std::make_integer_sequence<int, N>{}, f); }
}  // namespace p0

// ArFq with pass 0 compiled for the reference's (12289, 512) table: the two-operand product with the base
// multiplication only (serves).  Same stages, same bounds (fq_host.h: analyse32_bm_imm), 5 instructions per butterfly
// (fq_arith.cuh: mul_imm) and no constant loads.
struct ArFqImm : ArFq {
    static constexpr bool PASS0_IMM = true;
    template <int L, int M, bool BM> static constexpr bool serves() { return L == p0::kLogN && M == w32::FQ_POLYMUL && BM; }
    // stages 0..4 on x[m] = element tau + T m; x[0..15] arrive raw (load_operand)
    static __device__ __forceinline__ void fwd_pass0(u32 (&x)[32], const K &k)
    {
        const fq::ImmK kk{k.two23, k.q, k.nq};
        p0::static_for<5>([&](auto S) {
            constexpr int s = S, half = 16 >> s;
            p0::static_for<16>([&](auto J) {
                constexpr int m = (J / half) * 2 * half + J % half;
                constexpr fq::ImmTw t = fq::make_imm(p0::fwd((1 << s) + (m >> (5 - s))), p0::kQ);
                const u32 r = fq::mul_imm(x[m + half], t, 0u, kk);
                if constexpr (s == 0) {
                    // two opaque copies of kBias, as in ArFq::ct0: each result is one 3-input add
                    u32 kb1, kb2;
                    asm("mov.u32 %0, 0x4B400000;" : "=r"(kb1));
                    asm("mov.u32 %0, 1262485504;" : "=r"(kb2));
                    x[m + half] = x[m] - r + kb1;
                    x[m] = x[m] + r + kb2;
                } else {
                    x[m + half] = x[m] - r;
                    x[m] = x[m] + r;
                }
            });
        });
    }
    // stages 4..1 (biased products), then stage 0 with (n/4)^-1 folded into both branches; canonical residues out
    static __device__ __forceinline__ void inv_pass0(u32 (&x)[32], const K &k)
    {
        const fq::ImmK kk{k.two23, k.q, k.nq};
        p0::static_for<4>([&](auto I) {
            constexpr int s = 4 - I, half = 16 >> s;
            p0::static_for<16>([&](auto J) {
                constexpr int m = (J / half) * 2 * half + J % half;
                constexpr fq::ImmTw t = fq::make_imm(p0::inv((1 << s) + (m >> (5 - s))), p0::kQ);
                const u32 d = x[m] - x[m + half] + (u32)kBias;
                x[m] = x[m] + x[m + half] - (u32)kBias;
                x[m + half] = fq::mul_imm(d, t, (u32)kBias, kk);
            });
        });
        constexpr fq::ImmTw ni = fq::make_imm(p0::ninv(), p0::kQ), z = fq::make_imm(p0::inv1(), p0::kQ);
        p0::static_for<16>([&](auto M) {
            constexpr int m = M;
            const u32 s = x[m] + x[m + 16] - (u32)kBias;
            const u32 d = x[m] - x[m + 16] + (u32)kBias;
            const u32 ys = fq::mul_imm(s, ni, 0u, kk), yd = fq::mul_imm(d, z, 0u, kk);
            x[m] = min(ys, ys + (u32)k.q);
            x[m + 16] = min(yd, yd + (u32)k.q);
        });
    }
};
typedef w32::W32Const<ArFqImm> FqImmConst32;

// ---- key residues for the base-multiplication key product -------------------------------------------------------
// The key arrives fully transformed (the reference's NTT-domain order).  Two Gentleman-Sande stages and a factor 1/4
// take the four point values of block b back to the residue modulo X^4 - zeta_b; the table also holds zeta_b times
// the residue and float copies of both (fq_arith.cuh: basemul4_key).  One thread per block, 64-bit arithmetic: n/4
// threads per launch, negligible against the batch.  ktab (plan): [zi of stage logn-2 (n/4) | zi of stage logn-1
// (n/2) | zeta (n/4)], residues in [0, q).
template <class KT>
__global__ void k_key_residues(int32_t *__restrict__ kres, const KT *__restrict__ key, const int32_t *__restrict__ ktab,
                               int logn, int32_t q, int32_t inv4)
{
    const int n = 1 << logn, nb = n >> 2, T = n >> 5;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    auto modq = [q](long long v) { long long r = v % q; return r < 0 ? r + q : r; };
    long long v[4];
    for (int i = 0; i < 4; i++) {
        const unsigned pos = (unsigned)(4 * b + i);
        const unsigned idx = __brev(pos) >> (32 - logn);                  // reference index of internal position pos
        v[i] = modq((long long)key[idx]);
    }
    const long long zc = ktab[b], za = ktab[nb + 2 * b], zb_ = ktab[nb + 2 * b + 1], zeta = ktab[nb + 2 * nb + b];
    const long long u0 = v[0] + v[1], u1 = modq((v[0] - v[1]) * za), u2 = v[2] + v[3], u3 = modq((v[2] - v[3]) * zb_);
    long long r[4] = {u0 + u2, u1 + u3, modq((u0 - u2) * zc), modq((u1 - u3) * zc)};
    const int tau = b >> 3, j = b & 7;
    int32_t *o = kres + ((size_t)(4 * j) * T + tau) * 4;          // vector v of the block at o + 4 T v
    for (int i = 0; i < 4; i++) {
        long long x = modq(modq(r[i]) * inv4);
        long long z = modq(x * zeta);
        if (x > q / 2) x -= q;
        if (z > q / 2) z -= q;
        o[i] = (int32_t)x;
        o[4 * T + i] = __float_as_int((float)(int32_t)x);
        o[8 * T + i] = i ? (int32_t)z : 0;
        o[12 * T + i] = i ? __float_as_int((float)(int32_t)z) : 0;
    }
}

}  // namespace

struct Fq32State {
    int32_t *tab;                        // forward [w | wq | k | c], inverse [w | wq | k | c], n words each
    // degree-3 base multiplication of the two-operand product (fq_arith.cuh: basemul4); bm_ok == false: (q, n) outside
    // its bounds
    int32_t *zeta;                       // (w, wq) of zeta per block of four, [pair][tau][4 words]: n/2 words
    int32_t *ktab;                       // k_key_residues: [zi stage logn-2 | zi stage logn-1 | zeta], n words
    int32_t inv4;                        // 4^-1 mod q
    bool mv_ok, bm_ok;                   // mv_ok: mat-vec with up to 4 accumulated products
    bool imm;                            // the plan's pass-0 entries are ArFqImm's: its two-operand product runs that kernel
    FqConst32 prod, mv, bm;              // bm: last inverse stage with (n/4)^-1
    FqImmConst32 bm_imm;                 // bm for the ArFqImm kernel (the same words)
};

// true when the pass-0 entries of the base-multiplication constants are the ones compiled into ArFqImm and the
// interval analysis admits them as immediates
static bool imm_pass0_matches(const NttPlanDev &p, const FqConst32 &bm)
{
    if (p.rc.q != p0::kQ || p.logn != p0::kLogN) return false;
    int64_t w[64];
    for (int k = 1; k < 32; k++) {
        if (bm.f0[k - 1].w != p0::fwd(k) || (k > 1 && bm.i0[k - 1].w != p0::inv(k))) return false;
        w[2 * k - 2] = bm.f0[k - 1].w;
        w[2 * k - 1] = bm.i0[k - 1].w;
    }
    if (bm.i0[0].w != p0::inv1() || bm.ninv.w != p0::ninv()) return false;
    w[62] = bm.ninv.w;
    w[63] = bm.i0[0].w;
    int r0 = 0;
    return fq::analyse32_bm_imm(p.logn, p.rc.q, bm.x0, w, 64, &r0) && r0 == bm.r0;
}

int build_fq32_tables(NttPlanDev &p, const int32_t *w_host)
{
    if (p.logn < 8 || p.logn > 10) return SCGPU_OK;
    int r0 = 0; int32_t x0 = 0;
    if (!fq::analyse32(p.logn, p.rc.q, 1, &r0, &x0)) return SCGPU_OK;
    int r0_mv = 0; int32_t x0_mv = 0;
    const bool mv_ok = fq::analyse32(p.logn, p.rc.q, 4, &r0_mv, &x0_mv);     // up to 4 accumulated products
    std::vector<Tw> zf, zi;
    FqConst32 c;
    if (!fq::build_tables(p.logn, p.rc.q, w_host, zf, zi, c.ninv, c.one)) return SCGPU_OK;
    const int n = p.n;
    // forward [w | wq | k | c] then inverse [w | wq | k | c], n words each, entries of stages >= 5 thread-major
    std::vector<int32_t> pack(8 * n, 0);
    w32::pack_pass1<ArFq>(p.logn, zf, zi, [](const Tw &e, int k) {
        int32_t v;
        if (k == 0) v = e.w; else if (k == 1) memcpy(&v, &e.wq, 4); else if (k == 2) v = e.k; else memcpy(&v, &e.c, 4);
        return v;
    }, pack.data());
    Fq32State *s = p.fq32 = new Fq32State();
    s->mv_ok = mv_ok;
    SCGPU_CUDA_CHECK(cudaMalloc(&s->tab, sizeof(int32_t) * 8 * n));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->tab, pack.data(), sizeof(int32_t) * 8 * n, cudaMemcpyHostToDevice));
    // base multiplication of the two-operand product: zeta pairs thread-major, [pair pr][tau][w, wq, w, wq]
    // (blocks 8 tau + 2 pr and 8 tau + 2 pr + 1 of thread tau)
    int r0_bm = 0;
    Tw ninv_bm, i01_bm;
    const char *no_bm = getenv("SCGPU_NO_BASEMUL");
    if (!(no_bm && atoi(no_bm) != 0) && fq::analyse32_bm(p.logn, p.rc.q, x0, &r0_bm)) {
        std::vector<int32_t> zw; std::vector<float> zwq;
        fq::build_bm_tables(p.logn, p.rc.q, w_host, zw, zwq, ninv_bm, i01_bm);
        const int T = n / 32;
        std::vector<int32_t> zp((size_t)n / 2);
        for (int pr = 0; pr < 4; pr++)
            for (int tau = 0; tau < T; tau++)
                for (int u = 0; u < 2; u++) {
                    const int blk = 8 * tau + 2 * pr + u;
                    zp[((size_t)pr * T + tau) * 4 + 2 * u] = zw[blk];
                    memcpy(&zp[((size_t)pr * T + tau) * 4 + 2 * u + 1], &zwq[blk], 4);
                }
        SCGPU_CUDA_CHECK(cudaMalloc(&s->zeta, sizeof(int32_t) * zp.size()));
        SCGPU_CUDA_CHECK(cudaMemcpy(s->zeta, zp.data(), sizeof(int32_t) * zp.size(), cudaMemcpyHostToDevice));
        // table of k_key_residues: inverse twiddles of the last two stages (natural index) and zeta, in [0, q)
        std::vector<int32_t> kt((size_t)n);
        for (int b = 0; b < n / 4; b++) { kt[b] = zi[n / 4 + b].w; kt[n / 4 + n / 2 + b] = zw[b]; }
        for (int b = 0; b < n / 2; b++) kt[n / 4 + b] = zi[n / 2 + b].w;
        SCGPU_CUDA_CHECK(cudaMalloc(&s->ktab, sizeof(int32_t) * kt.size()));
        SCGPU_CUDA_CHECK(cudaMemcpy(s->ktab, kt.data(), sizeof(int32_t) * kt.size(), cudaMemcpyHostToDevice));
        s->inv4 = (int32_t)fq::powmod(4, p.rc.q - 2, p.rc.q);
        s->bm_ok = true;
    }
    c.pf = s->tab;
    c.pi = c.pf + 4 * n;
    c.pz = s->zeta;
    std::copy(zf.begin() + 1, zf.begin() + 32, c.f0);         // pass 0: entries 1..31
    std::copy(zi.begin() + 1, zi.begin() + 32, c.i0);
    c.q = p.rc.q; c.nq = -p.rc.q; c.x0 = x0;
    c.k.q = p.rc.q; c.k.nq = -p.rc.q;
    c.k.pwk = (int32_t)((uint32_t)kBias * (uint32_t)p.rc.q);
    c.k.invq = (float)(1.0 / (double)p.rc.q);
    c.k.pwb = (int32_t)((uint32_t)c.k.pwk + (uint32_t)kBias);
    c.k.two23 = 8388608.0f;
    c.M = (uint32_t)((1ull << 32) / (uint64_t)p.rc.q);
    s->prod = s->mv = s->bm = c;
    s->prod.r0 = r0;
    s->mv.r0 = r0_mv;
    if (s->bm_ok) {                                  // two inverse stages fewer: (n/4)^-1 in the last stage
        s->bm.r0 = r0_bm;
        s->bm.ninv = ninv_bm;
        s->bm.i0[0] = i01_bm;
        s->imm = imm_pass0_matches(p, s->bm);
        static_assert(sizeof(FqImmConst32) == sizeof(FqConst32) && std::is_trivially_copyable<FqConst32>::value, "same words");
        memcpy(&s->bm_imm, &s->bm, sizeof(FqConst32));
    }
    return SCGPU_OK;
}

void free_fq32_tables(NttPlanDev &p)
{
    if (!p.fq32) return;
    cudaFree(p.fq32->tab);
    cudaFree(p.fq32->zeta);
    cudaFree(p.fq32->ktab);
    delete p.fq32;
    p.fq32 = nullptr;
}

int fq32_matvec_lmax(const NttPlanDev &p) { return p.fq32 && p.fq32->mv_ok ? 4 : 0; }

// n = 256 (Kyber), l <= 4 (launch_matvec)
int launch_matvec_fq32(const NttPlanDev &p, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                       size_t count, cudaStream_t st, bool shared, const int32_t *e)
{
    return w32::launch_matvec_w32<ArFq>(p.fq32->mv, p.sm_count, out, A, s, k, l, count, st, !p.inputs_in_range, shared, e);
}

int launch_polymul_fq32(const NttPlanDev &p, int mode, int32_t *out, const int32_t *a, const void *b,
                        size_t b_stride, size_t count, cudaStream_t st, const int32_t *e)
{
    const Fq32State &fs = *p.fq32;
    if (b_stride == 0 && fs.bm_ok && (mode != w32::FQ_POLYMUL || count >= 64)) {
        // One second operand for the whole batch.  A shared key (the BLISS signing product) arrives transformed: its
        // residues modulo X^4 - zeta are prepared once for the launch in a stream-ordered scratch, then the batch runs
        // the base-multiplication key product.  A shared RAW operand (scgpu_polymul_batch with b_stride = 0) is first
        // taken to the reference's NTT domain by the canonical forward transform (one row) and is a shared key from
        // there on: the batch reads 8 n instead of 12 n bytes per product and transforms one operand instead of two.
        int32_t *kres = nullptr;
        SCGPU_CUDA_CHECK(cudaMallocAsync(reinterpret_cast<void **>(&kres), sizeof(int32_t) * 5 * (size_t)p.n, st));
        int32_t *hat = kres + 4 * (size_t)p.n;
        const unsigned nb = p.n / 4, th = 64;
        int r = SCGPU_OK;
        if (mode == w32::FQ_POLYMUL) {
            r = launch_ntt_fq32(p, 0, hat, static_cast<const int32_t *>(b), 1, st);
            b = hat;
        }
        if (r == SCGPU_OK) {
            if (mode == w32::FQ_KEY16)
                r = launch_kernel(k_key_residues<int16_t>, (nb + th - 1) / th, th, 0, st, kres, static_cast<const int16_t *>(b), fs.ktab, p.logn, p.rc.q, fs.inv4);
            else
                r = launch_kernel(k_key_residues<int32_t>, (nb + th - 1) / th, th, 0, st, kres, static_cast<const int32_t *>(b), fs.ktab, p.logn, p.rc.q, fs.inv4);
        }
        if (r == SCGPU_OK)
            r = w32::launch_polymul_w32<ArFq>(fs.bm, p.logn, p.sm_count, w32::FQ_KEYBM, out, a, kres, 0, count, st, true,
                                              !p.inputs_in_range, e);
        const cudaError_t fe = cudaFreeAsync(kres, st);
        if (r == SCGPU_OK && fe != cudaSuccess) { set_error("cudaFreeAsync failed: %s", cudaGetErrorString(fe)); r = SCGPU_ERR_CUDA; }
        return r;
    }
    const bool bm = mode == w32::FQ_POLYMUL && fs.bm_ok;
    if (bm && fs.imm)
        return w32::launch_polymul_w32<ArFqImm>(fs.bm_imm, p.logn, p.sm_count, mode, out, a, b, b_stride, count, st, true,
                                                !p.inputs_in_range, e);
    return w32::launch_polymul_w32<ArFq>(bm ? fs.bm : fs.prod, p.logn, p.sm_count, mode, out, a, b, b_stride, count, st, bm,
                                         !p.inputs_in_range, e);
}

int launch_ntt_fq32(const NttPlanDev &p, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t st)
{
    return w32::launch_ntt_w32<ArFq>(p.fq32->prod, p.logn, p.sm_count, inverse, out, a, count, st, !p.inputs_in_range);
}

}  // namespace scgpu
