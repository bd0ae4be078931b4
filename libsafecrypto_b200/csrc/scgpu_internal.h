// scgpu_internal.h -- shared between the translation units of libscgpu.so (not installed).
#pragma once
#include <vector>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>

#include "reduce.cuh"

namespace scgpu {

void set_error(const char *fmt, ...);
void count_launch();
int next_work_counter(cudaStream_t stream, unsigned long long **ctr, int chunk = 1);   // nullptr: static stride; chunk: groups per claim (1, 2, 4)
int init_work_counters();      // per-device ring of counters, allocated at plan creation

#define SCGPU_CUDA_CHECK(expr)                                                              \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ::scgpu::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return SCGPU_ERR_CUDA;                                                          \
        }                                                                                   \
    } while (0)

// Device-resident state of one (q, n, variant) parameter set.
struct NttPlanDev {
    int n, logn, variant, tw_bits, device;
    RedConst rc;
    int32_t *w;          // caller's w[n], sign-extended to 32 bits
    int32_t *r;          // caller's r[n]
    // fused-kernel constants (Montgomery domain, R = 2^32)
    MontTw *zeta_fwd;    // [n]: index 2^s + b  -> psi^brv(.) * R
    MontTw *zeta_inv;    // [n]: inverses, last-stage entries pre-multiplied by n^-1
    MontTw ninv;         // n^-1 * R   (sum branch of the last inverse stage)
    MontTw rsq;          // R^2 mod q  (brings one pointwise operand into Montgomery form)
    int32_t qinv;        // q^-1 mod 2^32
    int32_t fold;        // reserved
    int sm_count;
    // small-modulus fused kernels (32-bit Barrett, ntt_fast_sq.cu); sq_ok == 0: not applicable to (q, n)
    int sq_ok, sq_qbits, sq_r_pw, sq_r_inv[4], sq_r_inv_mv[4];
    int32_t *sq_zf, *sq_zi;
    int32_t sq_ninv, sq_x0;
    uint32_t sq_M;
    // small-modulus fused kernels, float-quotient arithmetic (ntt_fast_fq.cu); fq_ok == 0: not applicable
    int fq_ok, fq_r_inv[4], fq_r_inv_mv[4];
    int32_t fq_x0;
    void *fq_zf, *fq_zi;                 // int32 w[n] followed by float wq[n]
    alignas(16) unsigned char fq_ninv[16], fq_one[16];
    alignas(16) unsigned char fq_pass0[2 * 7 * 16];   // fq::Tw entries 1..7 of the forward / inverse table
    // warp-local 32-coefficient schedule of the same arithmetic (ntt_fast_fq32.cu)
    int fq32_ok, fq32_r0, fq32_mv_ok, fq32_r0_mv;
    int32_t fq32_x0;
    void *fq32_tab;                      // forward [w | wq | k | c], inverse [w | wq | k | c], n words each
    alignas(16) unsigned char fq32_pass0[2 * 31 * 16];
    // degree-3 base multiplication of the two-operand product (fq_arith.cuh: basemul4); 0: (q, n) outside its bounds
    int fq32_bm_ok, fq32_r0_bm;
    void *fq32_zeta;                     // (w, wq) of zeta per block of four, [pair][tau][4 words]: n/2 words
    void *fq32_ktab;                     // k_key_residues: [zi stage logn-2 | zi stage logn-1 | zeta], n words
    int32_t fq32_inv4;                   // 4^-1 mod q
    alignas(16) unsigned char fq32_ninv_bm[16], fq32_i01_bm[16];      // last inverse stage with (n/4)^-1
    int inputs_in_range;                 // SCGPU_PLAN_INPUTS_IN_RANGE: the fused products skip the range vote
    // Shoup / Montgomery arithmetic on the same schedule, for moduli up to 2^25 (ntt_fast_sh32.cu)
    int sh32_ok, sh32_r0, sh32_mv_ok, sh32_r0_mv;
    int sh32_mv_lmax;          // largest l whose exact 64-bit sums stay inside the Montgomery range (analyse_sh)
    int32_t sh32_x0;
    void *sh32_tab;                      // forward [w | wp], inverse [w | wp], n words each
    alignas(16) unsigned char sh32_pass0[2 * 31 * 8], sh32_ninv[8], sh32_one[8];
    alignas(16) unsigned char sh32_ninv_plain[8], sh32_zi1_plain[8];   // last-stage multipliers without the factor R
    // variant-exact transforms on the warp-local schedule (ntt_exact_w32.cu): 0 not applicable, 1 forward only (no r), 2 both
    int xw32_ok;
    int xw32_fpint;                      // fp / avx: the double quotient is evaluated in integers (ntt_exact_w32.cu header)
    void *xw32_tab;                      // [pass-1 w | aux | fwd twist w | aux | inv twist w | aux], n words each
    int32_t xw32_f0[62];                 // stages 0..4: 31 x w, 31 x aux
};

struct ExactArgs {
    int32_t *out;
    const void *a;
    const void *b;
    size_t b_stride;
    size_t count;
    const int32_t *w;
    const int32_t *r;
    int32_t *rcodes;
    RedConst rc;
    int op;
    int tw_bits;
    int32_t scalar;
};

int launch_exact(const NttPlanDev &plan, const ExactArgs &args, cudaStream_t stream);
// cdf_hp.cu: table of gauss_cdf_create_high_precision (host set-up): entries x precision/64 words, word 0 least significant
std::vector<uint64_t> build_cdf_high(int precision, int blinding, float tail, float sigma);
int launch_gen_rings(int prng_type, const uint8_t *seeds, size_t seed_len, size_t count, int32_t *out, int n, int k, int l,
                     int transpose, int32_t q, uint32_t q_bits, cudaStream_t stream);
int build_xw32_tables(NttPlanDev &plan, const int32_t *w_host, const int32_t *r_host);
void free_xw32_tables(NttPlanDev &plan);
int launch_exact_w32(const NttPlanDev &plan, int op, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_polymul(const NttPlanDev &plan, int32_t *out, const int32_t *a, const int32_t *b,
                   size_t b_stride, size_t count, cudaStream_t stream);
int launch_mul_key(const NttPlanDev &plan, int32_t *out, const int32_t *t, const void *key,
                   int key_bits, size_t key_stride, size_t count, cudaStream_t stream);
// shared: A is ONE matrix [k][l][n] for all `count` instances (scgpu_matvec_shared_batch)
int launch_matvec(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s,
                  int k, int l, size_t count, cudaStream_t stream, bool shared = false);
int build_fast_tables(NttPlanDev &plan, const int32_t *w_host);
void free_fast_tables(NttPlanDev &plan);
int set_force_montgomery(int on);
int set_fast_arith(int mode);           // 0 auto, 1 Montgomery, 2 Barrett-32, 3 float-quotient
int build_fq_tables(NttPlanDev &plan, const int32_t *w_host);
void free_fq_tables(NttPlanDev &plan);
int launch_polymul_fq(const NttPlanDev &plan, int mode, int32_t *out, const int32_t *a, const void *b,
                      size_t b_stride, size_t count, cudaStream_t stream);
int build_fq32_tables(NttPlanDev &plan, const int32_t *w_host);
void free_fq32_tables(NttPlanDev &plan);
int launch_polymul_fq32(const NttPlanDev &plan, int mode, int32_t *out, const int32_t *a, const void *b,
                        size_t b_stride, size_t count, cudaStream_t stream);
int build_sh32_tables(NttPlanDev &plan, const int32_t *w_host);
void free_sh32_tables(NttPlanDev &plan);
int launch_polymul_sh32(const NttPlanDev &plan, int mode, int32_t *out, const int32_t *a, const void *b,
                        size_t b_stride, size_t count, cudaStream_t stream);
int launch_matvec_sh32(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                       size_t count, cudaStream_t stream, bool shared = false);
int launch_ntt_fq32(const NttPlanDev &plan, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_ntt_sh32(const NttPlanDev &plan, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_ntt_canonical(const NttPlanDev &plan, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_matvec_fq32(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                       size_t count, cudaStream_t stream, bool shared = false);
int launch_matvec_fq(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                     size_t count, cudaStream_t stream, bool shared = false);
int build_sq_tables(NttPlanDev &plan, const int32_t *w_host);
void free_sq_tables(NttPlanDev &plan);
int launch_polymul_sq(const NttPlanDev &plan, int mode, int32_t *out, const int32_t *a, const void *b,
                      size_t b_stride, size_t count, cudaStream_t stream);
int launch_matvec_sq(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                     size_t count, cudaStream_t stream, bool shared = false);

}  // namespace scgpu
