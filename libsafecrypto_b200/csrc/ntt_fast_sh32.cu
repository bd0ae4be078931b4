// ntt_fast_sh32.cu -- fused negacyclic products for moduli the float-quotient arithmetic cannot serve
// (Dilithium's 8380417, 8399873: a 23-bit modulus leaves no room in a float mantissa), on the warp-local
// 32-coefficient schedule of warp32.cuh.
//
// Twiddle products are Shoup products: for a constant w (centred, |w| <= q/2) the table holds
// wp = round(w 2^32 / q); then  qe = hi32(x * wp),  t = x w - qe q  (IMAD.HI + 2 low IMADs, wrap-around
// arithmetic) lies in (-q/16, q + q/16) for |x| < 2^29: 8 fma-heavy clocks per butterfly instead of the 10 of
// the Montgomery product of ntt_fast.cu (2 x IMAD.HI + IMAD), one multiplication fewer on the critical path,
// and values need no domain conversion.  The n pointwise products of two variable operands are Montgomery
// products (a b R^-1, R = 2^32); the R is folded into the two multipliers of the last inverse stage.
// Coefficients are plain signed integers, lazily reduced; the host bounds every intermediate (analyse_sh).
#include "warp32.cuh"

#include <algorithm>
#include <vector>

namespace scgpu {

namespace {

using w32::u32;

struct ArSh {
    struct E { int32_t w, wp; };
    struct K { int32_t q, nq, qinv; };
    static constexpr bool BASEMUL = false;         // Montgomery pointwise products: no shared-quotient sums
    static constexpr bool STASH16 = false;          // mat-vec may keep the transformed vectors as int16
    static constexpr int WORDS = 2;
    static constexpr bool PASS0_IMM = false;
    template <int L, int M, bool BM> static constexpr bool serves() { return true; }
    static __device__ __forceinline__ u32 enc(int32_t x) { return (u32)x; }
    static __device__ __forceinline__ int32_t dec(u32 x) { return (int32_t)x; }
    static __device__ __forceinline__ u32 zero() { return 0u; }
    static __device__ __forceinline__ E cb(const E &e) { return e; }
    static __device__ __forceinline__ E mk(const int32_t (&w)[4]) { return E{w[0], w[1]}; }
    static __device__ __forceinline__ u32 mul(u32 x, const E &e, const K &k)
    {
        const int32_t qe = __mulhi((int32_t)x, e.wp);
        return x * (u32)e.w + (u32)qe * (u32)k.nq;
    }
    // forward butterfly in 4 instructions: the sum rides in the IMAD addend (lo + hi w - qe q), the difference is
    // 2 lo - sum (one IADD3)
    static __device__ __forceinline__ void ct(u32 &lo, u32 &hi, const E &z, const K &k)
    {
        const int32_t qe = __mulhi((int32_t)hi, z.wp);
        const u32 sum = (u32)qe * (u32)k.nq + (hi * (u32)z.w + lo);
        hi = lo + lo - sum;
        lo = sum;
    }
    static __device__ __forceinline__ void ct0(u32 &lo, u32 &hi, const E &z, const K &k) { ct(lo, hi, z, k); }   // enc is the identity
    static __device__ __forceinline__ void gs(u32 &lo, u32 &hi, const E &z, const K &k)
    {
        const u32 d = lo - hi;
        lo = lo + hi;
        hi = mul(d, z, k);
    }
    // products lie in (-q/16, q + q/16): one conditional +q, one conditional -q
    static __device__ __forceinline__ u32 canon(u32 y, const K &k)
    {
        y = min(y, y + (u32)k.q);
        return min(y, y - (u32)k.q);
    }
    static __device__ __forceinline__ void fin(u32 &lo, u32 &hi, const E &ninv, const E &z, const K &k)
    {
        const u32 s = lo + hi, d = lo - hi;
        lo = canon(mul(s, ninv, k), k);
        hi = canon(mul(d, z, k), k);
    }
    static __device__ __forceinline__ u32 red(u32 x, const E &one, const K &k) { return mul(x, one, k); }
    // a b R^-1 in (-q, q) for |a b| < q 2^31
    static __device__ __forceinline__ u32 mont(int32_t a, int32_t b, const K &k)
    {
        // low and high word by IMAD + IMAD.HI (3 issue units of the fma-heavy pipe; the 64-bit product as one
        // IMAD.WIDE measures 4.5, profiles/int_peaks_r02.txt -- the kernel is bound by that pipe, profiles/dil_polymul_r2_ncu.json)
        const u32 lo = (u32)a * (u32)b;
        const int32_t m = (int32_t)(lo * (u32)k.qinv);
        return (u32)(__mulhi(a, b) - __mulhi(m, k.q));
    }
    static __device__ __forceinline__ u32 pw(u32 a, u32 b, const K &k) { return mont((int32_t)a, (int32_t)b, k); }
    static __device__ __forceinline__ u32 pwraw(u32 a, int32_t kv, const K &k) { return mont((int32_t)a, kv, k); }
    // mat-vec accumulator: the l products of an output coefficient are summed EXACTLY in 64 bits (one IMAD.WIDE per
    // term) and reduced once -- |sum| < q 2^31 (analyse_sh), so one Montgomery step returns sum R^-1 in (-q, q).
    // (Before: a Montgomery product per term -- IMAD.WIDE + IMAD + IMAD.HI + 2 adds, 10 fma-heavy clocks instead of 4.)
    struct Acc { long long v; };
    static __device__ __forceinline__ Acc acc_zero() { return Acc{0ll}; }
    static __device__ __forceinline__ void acc_add(Acc &a, int32_t av, int32_t sv, const K &) { a.v += (long long)av * (long long)sv; }
    static __device__ __forceinline__ u32 acc_fin(const Acc &a, const K &k)
    {
        const int32_t m = (int32_t)((u32)a.v * (u32)k.qinv);
        return (u32)((int32_t)(a.v >> 32) - __mulhi(m, k.q));
    }
};

typedef w32::W32Const<ArSh> ShConst32;

int64_t powmod(int64_t b, int64_t e, int64_t q)
{
    __int128 r = 1, x = ((b % q) + q) % q;
    while (e > 0) { if (e & 1) r = (r * x) % q; x = (x * x) % q; e >>= 1; }
    return (int64_t)r;
}

ArSh::E make_entry(int64_t w, int64_t q)
{
    w = ((w % q) + q) % q;
    if (w > q / 2) w -= q;                                               // centred: |wp| < 2^31
    const __int128 num = (__int128)w * ((__int128)1 << 32);
    // round to nearest (floor of num / q + 1/2)
    __int128 wp = (2 * num + q) / (2 * q);
    if ((2 * num + q) % (2 * q) != 0 && (2 * num + q) < 0) wp -= 1;      // floor for negatives
    ArSh::E e;
    e.w = (int32_t)w;
    e.wp = (int32_t)wp;
    return e;
}

// |x w - qe q| <= q (1 + |x| 2^-33) + slack
double sh_bound(double b, double q) { return q * (1.0 + b / 8589934592.0) + 2.0; }

// Interval propagation over the schedule for this arithmetic; accumulate = pointwise products summed (mat-vec)
bool analyse_sh(int logn, int64_t qi, int accumulate, int *r0_out, int32_t *x0_out)
{
    if ((qi & 1) == 0 || qi < 257 || qi >= (1ll << 27)) return false;
    // up to 2^25: every value below 2^29 (quotient error < 1/16, the bound the kernels were first proven with); the 26-bit
    // moduli (Ring-TESLA's 51750913) use the whole signed range -- sh_bound() holds for any |x| < 2^31, the products stay
    // inside (-q, 2 q), which is all canon() needs
    const double q = (double)qi, lim = qi < (1ll << 25) ? 536870912.0 - 2.0 : 2147483648.0 - 67108864.0;
    const double x0 = 4.0 * q;
    double b = x0;
    for (int st = 0; st < logn; st++) {
        if (b >= lim) return false;
        b += sh_bound(b, q);
    }
    if (b >= lim) return false;
    double other = b > 32768.0 ? b : 32768.0;
    bool rb = false;
    if (b * other >= q * 2147483648.0) {                                 // Montgomery product range
        // reduce one operand first (bit 1 of the flag word): a Shoup product by 1 brings it to sh_bound(b)
        if (accumulate > 1) return false;
        rb = true;
        other = sh_bound(b, q) > 32768.0 ? sh_bound(b, q) : 32768.0;
        if (b * other >= q * 2147483648.0) return false;
    }
    // mat-vec: `accumulate` products of a matrix coefficient (|a| <= x0) and a transformed vector coefficient (<= b)
    // are summed in 64 bits and reduced once: the sum must stay inside the Montgomery range; the result is in (-q, q)
    if (accumulate > 1 && (double)accumulate * x0 * b >= q * 2147483648.0) return false;
    for (int r0 = 0; r0 <= 1; r0++) {
        double v = q;
        bool ok = true;
        for (int st = logn - 1; st >= 0 && ok; st--) {
            if (st == 4 && r0) { if (v >= lim) { ok = false; break; } v = sh_bound(v, q); }
            const double d = 2.0 * v;
            if (d >= lim) { ok = false; break; }
            const double prod = sh_bound(d, q);
            v = (st == 0) ? prod : (d > prod ? d : prod);
        }
        if (ok) { *r0_out = r0 | (rb ? 2 : 0); *x0_out = (int32_t)x0; return true; }
    }
    return false;
}

}  // namespace

struct Sh32State {
    int32_t *tab;                        // forward [w | wp], inverse [w | wp], n words each
    int mv_lmax;                         // largest l whose exact 64-bit sums stay inside the Montgomery range (analyse_sh)
    ShConst32 prod, mv;
    ShConst32 inv;                       // stand-alone inverse transform: last-stage multipliers without the factor R
};

int build_sh32_tables(NttPlanDev &p, const int32_t *w_host)
{
    if (p.logn < 8 || p.logn > 10) return SCGPU_OK;
    const int64_t q = p.rc.q;
    int r0 = 0; int32_t x0 = 0;
    if (!analyse_sh(p.logn, q, 1, &r0, &x0)) return SCGPU_OK;
    int r0_mv = 0; int32_t x0_mv = 0;
    const bool mv_ok = analyse_sh(p.logn, q, 4, &r0_mv, &x0_mv);
    // Dilithium's largest set is k = 6, l = 5 (240 q < 2^31 for q = 8380417): accept every l the sum bound admits
    int mv_lmax = mv_ok ? 4 : 0;
    for (int L = 5; L <= 8 && mv_ok; L++) {
        int r0x = 0; int32_t x0x = 0;
        if (!analyse_sh(p.logn, q, L, &r0x, &x0x) || r0x != r0_mv) break;
        mv_lmax = L;
    }
    const int n = p.n;
    const int64_t psi = (((int64_t)w_host[1] % q) + q) % q;
    if (powmod(psi, n, q) != q - 1) return SCGPU_OK;
    const int64_t R = (int64_t)((((__int128)1) << 32) % q);
    const int64_t ninvR = (int64_t)(((__int128)powmod(n, q - 2, q) * R) % q);     // Montgomery pointwise leaves R^-1
    std::vector<ArSh::E> zf(n, make_entry(1, q)), zi(n, make_entry(1, q));
    for (int k = 1; k < n; k++) {
        int e = 0;
        for (int b = 0; b < p.logn; b++) e |= ((k >> b) & 1) << (p.logn - 1 - b);
        const int64_t z = (((int64_t)w_host[e] % q) + q) % q;
        int64_t zinv = (q - (((int64_t)w_host[n - e] % q) + q) % q) % q;
        if (k == 1) zinv = (int64_t)(((__int128)zinv * ninvR) % q);
        zf[k] = make_entry(z, q);
        zi[k] = make_entry(zinv, q);
    }
    std::vector<int32_t> pack(4 * n, 0);
    w32::pack_pass1<ArSh>(p.logn, zf, zi, [](const ArSh::E &e, int k) { return k == 0 ? e.w : e.wp; }, pack.data());
    Sh32State *s = p.sh32 = new Sh32State();
    s->mv_lmax = mv_lmax;
    SCGPU_CUDA_CHECK(cudaMalloc(&s->tab, sizeof(int32_t) * 4 * n));
    SCGPU_CUDA_CHECK(cudaMemcpy(s->tab, pack.data(), sizeof(int32_t) * 4 * n, cudaMemcpyHostToDevice));
    uint32_t qinv = 1;
    for (int i = 0; i < 5; i++) qinv *= 2u - (uint32_t)q * qinv;         // Newton: q^-1 mod 2^32
    ShConst32 c;
    c.pf = s->tab;
    c.pi = c.pf + 2 * n;
    c.pz = nullptr;
    std::copy(zf.begin() + 1, zf.begin() + 32, c.f0);         // pass 0: entries 1..31
    std::copy(zi.begin() + 1, zi.begin() + 32, c.i0);
    c.ninv = make_entry(ninvR, q);
    c.one = make_entry(1, q);
    c.q = (int32_t)q; c.nq = (int32_t)-q; c.x0 = x0;
    c.k.q = (int32_t)q; c.k.nq = (int32_t)-q; c.k.qinv = (int32_t)qinv;
    c.M = (uint32_t)((1ull << 32) / (uint64_t)q);
    s->prod = s->mv = s->inv = c;
    s->prod.r0 = s->inv.r0 = r0;
    s->mv.r0 = r0_mv;
    // a stand-alone inverse transform has no Montgomery product to compensate: plain n^-1 and n^-1 psi^-(n/2)
    const int64_t nin = powmod(n, q - 2, q);
    const int e1 = 1 << (p.logn - 1);                                        // brv(1)
    const int64_t zinv1 = (q - (((int64_t)w_host[n - e1] % q) + q) % q) % q;
    s->inv.ninv = make_entry(nin, q);
    s->inv.i0[0] = make_entry((int64_t)(((__int128)zinv1 * nin) % q), q);
    return SCGPU_OK;
}

void free_sh32_tables(NttPlanDev &p)
{
    if (!p.sh32) return;
    cudaFree(p.sh32->tab);
    delete p.sh32;
    p.sh32 = nullptr;
}

int sh32_matvec_lmax(const NttPlanDev &p) { return p.sh32 ? p.sh32->mv_lmax : 0; }

// n = 256, l <= mv_lmax (launch_matvec)
int launch_matvec_sh32(const NttPlanDev &p, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                       size_t count, cudaStream_t st, bool shared, const int32_t *e)
{
    return w32::launch_matvec_w32<ArSh>(p.sh32->mv, p.sm_count, out, A, s, k, l, count, st, !p.inputs_in_range, shared, e);
}

int launch_polymul_sh32(const NttPlanDev &p, int mode, int32_t *out, const int32_t *a, const void *b,
                        size_t b_stride, size_t count, cudaStream_t st, const int32_t *e)
{
    return w32::launch_polymul_w32<ArSh>(p.sh32->prod, p.logn, p.sm_count, mode, out, a, b, b_stride, count, st, false,
                                         !p.inputs_in_range, e);
}

int launch_ntt_sh32(const NttPlanDev &p, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t st)
{
    return w32::launch_ntt_w32<ArSh>(inverse ? p.sh32->inv : p.sh32->prod, p.logn, p.sm_count, inverse, out, a, count, st,
                                     !p.inputs_in_range);
}

}  // namespace scgpu
