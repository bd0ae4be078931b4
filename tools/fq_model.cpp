// fq_model.cpp -- CPU model of the float-quotient kernels' arithmetic (fq_arith.cuh, fq_host.h): runs the same
// stage structure with the same twiddle entries, compares with a schoolbook negacyclic product and checks
// the analysed bounds.   g++ -O2 -std=c++17 -I libsafecrypto_b200/csrc tools/fq_model.cpp -o /tmp/fq_model
#include "fq_host.h"
#include <cstdio>
#include <cstdlib>
#include <random>
using namespace scgpu::fq;

static double g_max_fwd, g_max_inv, g_max_fin;
static int32_t rd(int32_t xb, double &mx) { double a = fabs((double)(xb - kBias)); if (a > mx) mx = a; return xb; }

static int g_r0 = -1;      // >= 0: warp-local schedule (one optional reduction before stage 4) instead of sc.r_inv
static void polymul(int logn, int64_t q, const std::vector<Tw> &zf, const std::vector<Tw> &zi, const Tw &ninv, const Tw &one,
                    const Schedule &sc, const int32_t *a, const int32_t *b, int32_t *out)
{
    const int n = 1 << logn; const int32_t nq = (int32_t)-q;
    std::vector<int32_t> x[2]; x[0].resize(n); x[1].resize(n);
    for (int i = 0; i < n; i++) { x[0][i] = a[i] + kBias; x[1][i] = b[i] + kBias; }
    for (int op = 0; op < 2; op++)
        for (int s = 0; s < logn; s++) {
            const int len = n >> (s + 1);
            for (int blk = 0; blk < (1 << s); blk++)
                for (int j = 0; j < len; j++) {
                    int32_t &lo = x[op][2 * blk * len + j], &hi = x[op][2 * blk * len + j + len];
                    int32_t t = mul(rd(hi, g_max_fwd), zf[(1 << s) + blk], nq);
                    hi = lo - t; lo = lo + t;
                }
        }
    const float invq = (float)(1.0 / (double)q);
    const int32_t pwk = (int32_t)((uint32_t)kBias * (uint32_t)q);
    std::vector<int32_t> y(n);
    for (int i = 0; i < n; i++) y[i] = mul_var(x[0][i] - kBias, x[1][i] - kBias, invq, pwk, nq) + kBias;
    const int npass = (logn + 2) / 3;
    for (int s = logn - 1; s >= 0; s--) {
        const int len = n >> (s + 1);
        // reduce at the entry of a pass (first stage the pass executes is its highest stage index)
        for (int p = 0; p < npass && g_r0 < 0; p++) {
            const int J = (logn - 3 * p) >= 3 ? 3 : (logn - 3 * p);
            if (s == 3 * p + J - 1 && sc.r_inv[p]) for (int i = 0; i < n; i++) y[i] = mul(rd(y[i], g_max_inv), one, nq);
        }
        if (g_r0 == 1 && s == 4) for (int i = 0; i < n; i++) y[i] = mul(rd(y[i], g_max_inv), one, nq);
        for (int blk = 0; blk < (1 << s); blk++)
            for (int j = 0; j < len; j++) {
                int32_t &lo = y[2 * blk * len + j], &hi = y[2 * blk * len + j + len];
                int32_t sb = lo + hi - kBias, db = lo - hi + kBias;
                if (s == 0) {
                    lo = mul(rd(sb, g_max_inv), ninv, nq); hi = mul(rd(db, g_max_inv), zi[1], nq);
                    if (fabs((double)lo) > g_max_fin) g_max_fin = fabs((double)lo);
                    if (fabs((double)hi) > g_max_fin) g_max_fin = fabs((double)hi);
                    lo += (lo >> 31) & (int32_t)q; hi += (hi >> 31) & (int32_t)q;
                } else {
                    hi = mul(rd(db, g_max_inv), zi[(1 << s) + blk], nq); lo = sb;
                }
            }
    }
    for (int i = 0; i < n; i++) out[i] = y[i];
}

// warp-local schedule with the degree-3 base multiplication (fq_arith.cuh: basemul4)
static double g_max_sum;
// imm: stages 0..4 of both directions with the entries as instruction immediates (fq_arith.cuh: mul_imm), as the
// kernel compiled for the reference's (12289, 512) table runs them
static void polymul_bm(int logn, int64_t q, const std::vector<Tw> &zf, const std::vector<Tw> &zi, const Tw &one, int r0,
                       const int32_t *a, const int32_t *b, int32_t *out, const int32_t *w_host, bool imm = false)
{
    const ImmK kk{8388608.0f, (int32_t)q, (int32_t)-q};
    const int n = 1 << logn; const int32_t nq = (int32_t)-q;
    std::vector<int32_t> zw; std::vector<float> zwq; Tw ninv_bm, i01_bm;
    build_bm_tables(logn, q, w_host, zw, zwq, ninv_bm, i01_bm);
    std::vector<int32_t> x[2]; x[0].resize(n); x[1].resize(n);
    for (int i = 0; i < n; i++) { x[0][i] = a[i] + kBias; x[1][i] = b[i] + kBias; }
    for (int op = 0; op < 2; op++)
        for (int s = 0; s < logn - 2; s++) {
            const int len = n >> (s + 1);
            for (int blk = 0; blk < (1 << s); blk++)
                for (int j = 0; j < len; j++) {
                    int32_t &lo = x[op][2 * blk * len + j], &hi = x[op][2 * blk * len + j + len];
                    int32_t t = imm && s < 5 ? (int32_t)mul_imm((uint32_t)rd(hi, g_max_fwd), make_imm(zf[(1 << s) + blk].w, q), 0u, kk)
                                             : mul(rd(hi, g_max_fwd), zf[(1 << s) + blk], nq);
                    hi = lo - t; lo = lo + t;
                    if (s == logn - 3) { hi -= kBias; lo -= kBias; }         // the last stage emits unbiased values
                }
        }
    const float invq = (float)(1.0 / (double)q);
    const int32_t pwk = (int32_t)((uint32_t)kBias * (uint32_t)q);
    const int32_t pwb = (int32_t)((uint32_t)pwk + (uint32_t)kBias);
    std::vector<int32_t> y(n);
    for (int blk = 0; blk < n / 4; blk++) {
        int32_t aa[4], bb[4], cc[4];
        for (int i = 0; i < 4; i++) {
            aa[i] = x[0][4 * blk + i]; bb[i] = x[1][4 * blk + i];
            if (fabs((double)aa[i]) > g_max_fwd) g_max_fwd = fabs((double)aa[i]);
            if (fabs((double)bb[i]) > g_max_fwd) g_max_fwd = fabs((double)bb[i]);
        }
        basemul4(cc, aa, bb, zw[blk], zwq[blk], invq, pwk, pwb, nq);
        for (int i = 0; i < 4; i++) { y[4 * blk + i] = cc[i]; double m = fabs((double)(cc[i] - kBias)); if (m > g_max_sum) g_max_sum = m; }
    }
    for (int s = logn - 3; s >= 0; s--) {
        const int len = n >> (s + 1);
        if (r0 == 1 && s == 4) for (int i = 0; i < n; i++) y[i] = mul(rd(y[i], g_max_inv), one, nq);
        for (int blk = 0; blk < (1 << s); blk++)
            for (int j = 0; j < len; j++) {
                int32_t &lo = y[2 * blk * len + j], &hi = y[2 * blk * len + j + len];
                int32_t sb = lo + hi - kBias, db = lo - hi + kBias;
                if (s == 0) {
                    if (imm) {
                        lo = (int32_t)mul_imm((uint32_t)rd(sb, g_max_inv), make_imm(ninv_bm.w, q), 0u, kk);
                        hi = (int32_t)mul_imm((uint32_t)rd(db, g_max_inv), make_imm(i01_bm.w, q), 0u, kk);
                    } else {
                        lo = mul(rd(sb, g_max_inv), ninv_bm, nq); hi = mul(rd(db, g_max_inv), i01_bm, nq);
                    }
                    if (fabs((double)lo) > g_max_fin) g_max_fin = fabs((double)lo);
                    if (fabs((double)hi) > g_max_fin) g_max_fin = fabs((double)hi);
                    lo += (lo >> 31) & (int32_t)q; hi += (hi >> 31) & (int32_t)q;
                } else {
                    hi = imm && s < 5 ? (int32_t)mul_imm((uint32_t)rd(db, g_max_inv), make_imm(zi[(1 << s) + blk].w, q), (uint32_t)kBias, kk)
                                      : mul(rd(db, g_max_inv), zi[(1 << s) + blk], nq);
                    lo = sb;
                }
            }
    }
    for (int i = 0; i < n; i++) out[i] = y[i];
}

static void school(int n, int64_t q, const int32_t *a, const int32_t *b, int32_t *out)
{
    std::vector<int64_t> acc(n, 0);
    for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) {
        int64_t p = ((int64_t)a[i] % q) * ((int64_t)b[j] % q) % q;
        int k = i + j;
        if (k >= n) { k -= n; p = -p; }
        acc[k] = (acc[k] + p) % q;
    }
    for (int i = 0; i < n; i++) out[i] = (int32_t)((acc[i] % q + q) % q);
}

int main()
{
    struct { int logn; int64_t q; } sets[] = {{9, 12289}, {10, 12289}, {8, 7681}, {8, 12289}, {10, 18433}, {9, 40961}, {10, 61441}, {8, 257 * 512 + 1}};
    std::mt19937 rng(7);
    int bad = 0;
    for (auto &ps : sets) {
        const int logn = ps.logn, n = 1 << logn; const int64_t q = ps.q;
        int64_t g = 2; while (g < q && powmod(g, n, q) != q - 1) g++;
        if (g >= q) { printf("q=%lld n=%d: no 2n-th root\n", (long long)q, n); continue; }
        std::vector<int32_t> w(n); int64_t c = 1; for (int i = 0; i < n; i++) { w[i] = (int32_t)c; c = c * g % q; }
        std::vector<Tw> zf, zi; Tw ninv, one;
        Schedule sc = analyse(logn, q, 1);
        printf("q=%lld n=%d ok=%d r_inv=%d%d%d%d x0=%d fwd_max=%.0f inv_max=%.0f final=%.0f\n", (long long)q, n, sc.ok, sc.r_inv[0], sc.r_inv[1], sc.r_inv[2], sc.r_inv[3], sc.x0, sc.fwd_max, sc.inv_max, sc.final_max);
        if (!sc.ok) continue;
        if (!build_tables(logn, q, w.data(), zf, zi, ninv, one)) { printf("  tables failed\n"); bad++; continue; }
        std::vector<int32_t> a(n), b(n), o(n), e(n);
        const int x0 = sc.x0;
        for (int sched = 0; sched < 4; sched++) {
        g_max_fwd = g_max_inv = g_max_fin = g_max_sum = 0;
        g_r0 = -1;
        BmBounds bmb; int r0bm = 0;
        if (sched == 3) {
            // the pass-0 entries as immediates: the 62 entries of stages 0..4 and the two of the last stage
            std::vector<int32_t> zw; std::vector<float> zwq; Tw nb, ib;
            build_bm_tables(logn, q, w.data(), zw, zwq, nb, ib);
            std::vector<int64_t> ent;
            for (int k = 1; k < 32; k++) { ent.push_back(zf[k].w); if (k > 1) ent.push_back(zi[k].w); }
            ent.push_back(nb.w); ent.push_back(ib.w);
            if (!analyse32_bm_imm(logn, q, x0, ent.data(), (int)ent.size(), &r0bm)) { printf("  pass 0 with immediate entries: refused\n"); continue; }
            analyse32_bm(logn, q, x0, &r0bm, &bmb);
            printf("  pass 0 with immediate entries: accepted r0=%d\n", r0bm);
        }
        if (sched == 2) {
            if (!analyse32_bm(logn, q, x0, &r0bm, &bmb)) { printf("  base multiplication: not applicable\n"); continue; }
            printf("  warp-local schedule with base multiplication: r0=%d fwd_max=%.0f pw_max=%.0f\n", r0bm, bmb.fwd_max, bmb.pw_max);
        }
        if (sched == 1) {
            int r0 = 0; int32_t x032 = 0;
            if (!analyse32(logn, q, 1, &r0, &x032)) { printf("  warp-local schedule: not applicable\n"); continue; }
            g_r0 = r0;
            printf("  warp-local schedule: r0=%d\n", r0);
        }
        for (int trial = 0; trial < 60; trial++) {
            for (int i = 0; i < n; i++) {
                switch (trial % 6) {
                case 0: a[i] = rng() % q; b[i] = rng() % q; break;
                case 1: a[i] = (int32_t)(rng() % (2 * x0 + 1)) - x0; b[i] = (int32_t)(rng() % (2 * x0 + 1)) - x0; break;
                case 2: a[i] = x0; b[i] = (i & 1) ? -x0 : x0; break;
                case 3: a[i] = (rng() & 1) ? x0 : -x0; b[i] = (rng() & 1) ? x0 : -x0; break;
                case 4: a[i] = (i == (int)(rng() % n)) ? x0 : 0; b[i] = -x0; break;
                default: a[i] = (int32_t)(q - 1); b[i] = (int32_t)(q - 1); break;
                }
            }
            if (sched >= 2) polymul_bm(logn, q, zf, zi, one, r0bm, a.data(), b.data(), o.data(), w.data(), sched == 3);
            else polymul(logn, q, zf, zi, ninv, one, sc, a.data(), b.data(), o.data());
            school(n, q, a.data(), b.data(), e.data());
            for (int i = 0; i < n; i++) if (o[i] != e[i]) { if (bad < 5) printf("  MISMATCH trial %d i=%d got %d want %d\n", trial, i, o[i], e[i]); bad++; break; }
        }
        printf("  observed: fwd %.0f inv %.0f final %.0f  (limit %d)\n", g_max_fwd, g_max_inv, g_max_fin, kLimit);
        if (sched >= 2 && (g_max_fwd > bmb.fwd_max || g_max_sum > bmb.pw_max)) { printf("  BOUND VIOLATED (base multiplication: fwd %.0f pw %.0f)\n", g_max_fwd, g_max_sum); bad++; }
        if (g_max_fwd > sc.fwd_max || g_max_inv >= (double)kLimit || g_max_fin >= (double)q) { printf("  BOUND VIOLATED\n"); bad++; }
        if (sched == 0 && (g_max_inv > sc.inv_max || g_max_fin > sc.final_max)) { printf("  BOUND VIOLATED (8-coefficient schedule)\n"); bad++; }
        }
    }
    printf(bad ? "FAIL %d\n" : "ALL OK\n", bad);
    return bad != 0;
}
