// fq_host.h -- host-side set-up of the float-quotient kernels: twiddle entries and the interval analysis
// that proves every value read as a float stays below 2^22 and the final residue lies in (-q, q).
// Plain C++ (no CUDA) so that tools/fq_model.cpp can run the same code on the CPU.
#pragma once
#include "fq_arith.cuh"

#include <vector>

namespace scgpu {
namespace fq {

struct Schedule {
    int ok;             // 0: (q, n) cannot be served by this arithmetic
    int r_inv[4];       // reduce all slots at the entry of inverse pass p (pass 0 holds the final stage)
    int32_t x0;         // |input| bound of the fast path
    double fwd_max;     // proven bounds (for the model's assertions)
    double inv_max;
    double final_max;
};

inline int64_t powmod(int64_t b, int64_t e, int64_t q)
{
    __int128 r = 1, x = ((b % q) + q) % q;
    while (e > 0) { if (e & 1) r = (r * x) % q; x = (x * x) % q; e >>= 1; }
    return (int64_t)r;
}

// entry for multiplication by w (any representative), result biased when out_biased
inline Tw make_tw(int64_t w, int64_t q, bool out_biased)
{
    Tw t;
    w = ((w % q) + q) % q;
    const int64_t k22 = (w * (1ll << 23) + q) / (2 * q);             // round(w * 2^22 / q)
    t.w = (int32_t)w;
    t.wq = (float)((double)k22 / 4194304.0);                         // k22 <= 2^22: exact
    t.c = (float)(12582912.0 - 3.0 * (double)k22);                   // integer in [0, 2^24): exact
    uint32_t k = (uint32_t)kBias * (uint32_t)q - (uint32_t)kBias * (uint32_t)w;
    if (out_biased) k += (uint32_t)kBias;
    t.k = (int32_t)k;
    return t;
}

// |x w - qe q| for |x| <= b  (+1 of slack for the rounding of the bound itself)
inline double mul_bound(double b, double q) { return q * (0.5 + b / 8388608.0) + 1.0; }

// Interval propagation over the kernels' dataflow; `accumulate` = number of pointwise products summed before
// the inverse transform (1: polymul / key product, l: mat-vec).  key_max = largest |second operand| of a
// key product (SINT16 keys: 32768).
inline Schedule analyse(int logn, int64_t qi, int accumulate)
{
    Schedule s;
    s.ok = 0;
    for (int i = 0; i < 4; i++) s.r_inv[i] = 0;
    const double q = (double)qi, lim = (double)kLimit - 2.0;
    s.x0 = (int32_t)(4 * qi);
    if (qi < 257 || qi >= (1 << 18) || (qi & 1) == 0) return s;
    // forward: one product per stage on the difference branch, additive growth
    double b = (double)s.x0;
    for (int st = 0; st < logn; st++) {
        if (b >= lim) return s;
        b += mul_bound(b, q);
    }
    s.fwd_max = b;
    if (b >= lim) return s;
    // pointwise: |a b| / q < 2^22 with both operands at the forward bound, or one at max(q, 32768)
    const double other = b > 32768.0 ? b : 32768.0;
    const double quo = b * other / q;
    if (quo >= lim) return s;
    const double pw = q * (0.5 + 2.0 * quo / 16777216.0) + 2.0;       // roundings: g, 1/q (2^-24 relative each), the FMA (1/2)
    // inverse passes: pass np-1 first; slots m = 0..7, stage distance 1, 2, 4 in slot units
    const int npass = (logn + 2) / 3;
    double bin = pw * accumulate;
    s.inv_max = bin;
    for (int pass = npass - 1; pass >= 0; pass--) {
        const int J = (logn - 3 * pass) >= 3 ? 3 : (logn - 3 * pass);
        int chosen = -1;
        double bout = 0, seen = 0, fin = 0;
        for (int r = 0; r <= 1 && chosen < 0; r++) {
            double v[8];
            if (r && bin >= lim) break;
            for (int m = 0; m < 8; m++) v[m] = r ? mul_bound(bin, q) : bin;
            bool ok = true;
            seen = 0; fin = 0;
            for (int st = 0; st < J && ok; st++) {
                const int delta = 1 << st;
                const bool last = (pass == 0 && st == J - 1);
                for (int m = 0; m < 8 && ok; m++) {
                    if (m & delta) continue;
                    const double d = v[m] + v[m + delta];
                    if (d >= lim) { ok = false; break; }
                    seen = d > seen ? d : seen;
                    v[m + delta] = mul_bound(d, q);
                    v[m] = last ? mul_bound(d, q) : d;
                    if (last) fin = v[m] > fin ? v[m] : fin;
                }
            }
            if (ok && pass == 0 && fin >= q) ok = false;          // canonicalisation adds q at most once
            if (ok) {
                chosen = r;
                for (int m = 0; m < 8; m++) bout = v[m] > bout ? v[m] : bout;
            }
        }
        if (chosen < 0) return s;
        s.r_inv[pass] = chosen;
        s.inv_max = seen > s.inv_max ? seen : s.inv_max;
        if (pass == 0) s.final_max = fin;
        bin = bout;
    }
    s.ok = 1;
    return s;
}

// Bounds of the warp-local 32-coefficient schedule (ntt_fast_fq32.cu): forward and pointwise as in analyse; inverse: sums double per stage, products
// are bounded by mul_bound; one optional reduction of every coefficient between the two inverse passes.
inline bool analyse32(int logn, int64_t qi, int accumulate, int *r0_out, int32_t *x0_out)
{
    const Schedule s = analyse(logn, qi, 1);        // forward + pointwise part (and q range checks)
    if (!s.ok) return false;
    const double q = (double)qi, lim = (double)kLimit - 2.0;
    const double other = s.fwd_max > 32768.0 ? s.fwd_max : 32768.0;
    const double quo = s.fwd_max * other / q;
    double pw = q * (0.5 + 2.0 * quo / 16777216.0) + 2.0;
    if (accumulate > 1) {
        // mat-vec (ArFq::Acc): the products of an output coefficient, |a| <= x0 times |s| <= fwd_max each, share
        // one quotient: the summed quotient must stay in the magic-number range, and the float sum adds
        // accumulate roundings of half an ulp of the largest partial sum
        const double sum = accumulate * (double)s.x0 * s.fwd_max;
        if (sum / q >= lim) return false;
        const double ulp = std::ldexp(1.0, std::ilogb(sum) - 23);
        pw = q * (0.5 + 2.0 * (sum / q) / 16777216.0) + accumulate * ulp + 2.0;
        accumulate = 1;
    }
    for (int r0 = 0; r0 <= 1; r0++) {
        double b = pw * accumulate;
        bool ok = true;
        for (int st = logn - 1; st >= 0 && ok; st--) {
            if (st == 4 && r0) { if (b >= lim) { ok = false; break; } b = mul_bound(b, q); }
            const double d = 2.0 * b;                        // |lo + hi|, |lo - hi|
            if (d >= lim) { ok = false; break; }
            const double prod = mul_bound(d, q);
            if (st == 0) { if (prod >= q) ok = false; b = prod; }
            else b = d > prod ? d : prod;
        }
        if (ok) { *r0_out = r0; *x0_out = s.x0; return true; }
    }
    return false;
}

// Bounds of the warp-local schedule with the degree-3 base multiplication (fq_arith.cuh: basemul4): logn - 2
// forward stages, n/4 products modulo X^4 - zeta, logn - 2 inverse stages.  x0 = |input| bound.
struct BmBounds { double fwd_max, sum_max, pw_max; };
inline bool analyse32_bm(int logn, int64_t qi, int32_t x0, int *r0_out, BmBounds *bounds = nullptr)
{
    const double q = (double)qi, lim = (double)kLimit - 2.0;
    if (qi < 257 || qi >= (1 << 18) || (qi & 1) == 0 || logn < 8) return false;
    double b = (double)x0;
    for (int st = 0; st < logn - 2; st++) {
        if (b >= lim) return false;
        b += mul_bound(b, q);
    }
    if (b >= lim) return false;                                  // read as a float by the conversions
    const double zb = mul_bound(b, q);                           // |zeta a_i|
    const double big = b > zb ? b : zb;
    const double sum = 4.0 * big * b;                            // four products per output coefficient
    if (sum / q >= lim) return false;
    // the float sum: one rounding per term, each at most half an ulp of a partial sum below `sum`; 1/q is rounded
    // (2^-24 relative); the FMA that adds the magic number rounds to an integer (1/2)
    double ferr = 0;
    for (int t = 1; t <= 4; t++) ferr += 0.5 * std::ldexp(1.0, std::ilogb(t * big * b) - 23);   // partial sum of t terms
    const double pw = q * (0.5 + 2.0 * (sum / q) / 16777216.0) + ferr + 2.0;
    if (bounds) { bounds->fwd_max = b; bounds->sum_max = sum; bounds->pw_max = pw; }
    for (int r0 = 0; r0 <= 1; r0++) {
        double v = pw;
        bool ok = true;
        for (int st = logn - 3; st >= 0 && ok; st--) {
            if (st == 4 && r0) { if (v >= lim) { ok = false; break; } v = mul_bound(v, q); }
            const double d = 2.0 * v;
            if (d >= lim) { ok = false; break; }
            const double prod = mul_bound(d, q);
            if (st == 0) { if (prod >= q) ok = false; v = prod; }
            else v = d > prod ? d : prod;
        }
        if (ok) { *r0_out = r0; return true; }
    }
    return false;
}

// The same schedule with the pass-0 entries as instruction immediates (fq_arith.cuh: make_imm, mul_imm).  A product by an immediate entry has the error bound of mul (|qe - x a / q| <= 1/2 + |x| 2^-23), so the
// bounds of analyse32_bm hold unchanged; what is new is that its FFMA must stay inside the binade [2^23, 2^24) for
// every entry w[0 .. count) and every value analyse32_bm admits (|x| < lim):  0 <= wq (3 2^22 - lim)  and
// 2^23 + wq (3 2^22 + lim) <= 2^24 - 1.
inline bool analyse32_bm_imm(int logn, int64_t qi, int32_t x0, const int64_t *w, int count, int *r0_out)
{
    if (!analyse32_bm(logn, qi, x0, r0_out)) return false;
    const double lim = (double)kLimit - 2.0;
    for (int i = 0; i < count; i++) {
        const double wq = (double)make_imm(w[i], qi).wq;
        if (wq * (12582912.0 - lim) < 0.0 || 8388608.0 + wq * (12582912.0 + lim) > 16777215.0) return false;
    }
    return true;
}

// zeta_b = zf[n/4 + b]^2 (the modulus X^4 - zeta_b of block b after stage logn - 3) as (w, wq) pairs, and the two
// entries of the last inverse stage with (n/4)^-1 instead of n^-1 (two Gentleman-Sande stages fewer double the
// result twice less)
inline void build_bm_tables(int logn, int64_t q, const int32_t *w_host, std::vector<int32_t> &zeta_w,
                            std::vector<float> &zeta_wq, Tw &ninv_bm, Tw &i01_bm)
{
    const int n = 1 << logn, nb = n / 4;
    zeta_w.resize(nb); zeta_wq.resize(nb);
    for (int b = 0; b < nb; b++) {
        const int k = nb + b;
        int e = 0;
        for (int t = 0; t < logn; t++) e |= ((k >> t) & 1) << (logn - 1 - t);
        const int64_t z = (((int64_t)w_host[e] % q) + q) % q;
        const Tw tw = make_tw((int64_t)(((__int128)z * z) % q), q, false);
        zeta_w[b] = tw.w; zeta_wq[b] = tw.wq;
    }
    const int64_t nin4 = powmod(n / 4, q - 2, q);
    const int64_t zinv1 = (q - (((int64_t)w_host[n - n / 2] % q) + q) % q) % q;       // zi[1] without n^-1 (brv(1) = n/2)
    ninv_bm = make_tw(nin4, q, false);
    i01_bm = make_tw((int64_t)(((__int128)zinv1 * nin4) % q), q, false);
}

// zf[k] = psi^brv(k) (k = 2^s + b: stage s, block b); zi[k] = its inverse, zi[1] also carries n^-1.
// Forward products and the two final-stage products are unbiased, every other inverse product is biased.
inline bool build_tables(int logn, int64_t q, const int32_t *w_host, std::vector<Tw> &zf, std::vector<Tw> &zi,
                         Tw &ninv, Tw &one)
{
    const int n = 1 << logn;
    const int64_t psi = (((int64_t)w_host[1] % q) + q) % q;
    if (powmod(psi, n, q) != q - 1) return false;
    const int64_t nin = powmod(n, q - 2, q);
    zf.assign(n, make_tw(1, q, false));
    zi.assign(n, make_tw(1, q, true));
    for (int k = 1; k < n; k++) {
        int e = 0;
        for (int b = 0; b < logn; b++) e |= ((k >> b) & 1) << (logn - 1 - b);
        const int64_t z = (((int64_t)w_host[e] % q) + q) % q;
        int64_t zinv = (q - (((int64_t)w_host[n - e] % q) + q) % q) % q;
        if (k == 1) zinv = (int64_t)(((__int128)zinv * nin) % q);
        zf[k] = make_tw(z, q, false);
        zi[k] = make_tw(zinv, q, k != 1);
    }
    ninv = make_tw(nin, q, false);
    one = make_tw(1, q, true);
    return true;
}

}  // namespace fq
}  // namespace scgpu
