// scgpu_internal.h -- shared between the translation units of libscgpu.so (not installed).
#pragma once
#include <vector>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>
#include <type_traits>
#include <utility>

#include "reduce.cuh"
#include "../../include/scgpu.h"

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

// One kernel launch: the 200 KiB opt-in for a kernel with dynamic shared memory (per launch, not once: the attribute
// belongs to the current device's context and plans exist per device), the launch, the launch count, the error check.
template <class... P, class... A>
int launch_kernel(void (*kernel)(P...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, A &&...args)
{
    if (smem > 0) SCGPU_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    kernel<<<grid, block, smem, st>>>(std::forward<A>(args)...);
    count_launch();
    SCGPU_CUDA_CHECK(cudaGetLastError());
    return SCGPU_OK;
}

// Run-time choices to template arguments.  with_int<Vs...>(v, f): f(std::integral_constant<int, v>{}) for the listed
// value v (SCGPU_ERR_UNSUPPORTED for any other); with_flags(f, b0, b1, ...): f(std::bool_constant<b0>{}, ...).
template <int... Vs, class F>
int with_int(int v, F &&f)
{
    int r = SCGPU_ERR_UNSUPPORTED;
    (void)((v == Vs ? (r = f(std::integral_constant<int, Vs>{}), true) : false) || ...);
    return r;
}
template <class F>
int with_flags(F &&f) { return f(); }
template <class F, class... B>
int with_flags(F &&f, bool b, B... rest)
{
    if (b) return with_flags([&](auto... t) { return f(std::true_type{}, t...); }, rest...);
    return with_flags([&](auto... t) { return f(std::false_type{}, t...); }, rest...);
}

// Plan state of each arithmetic of the fused and warp-local kernels, defined in its own .cu: device tables, the
// kernel-constant structs its launches pass (built once at plan creation, read-only afterwards: plans are shared by
// host threads) and what the arithmetic can serve.
struct MontState;      // ntt_fast.cu: Montgomery, any odd q < 2^30
struct SqState;        // ntt_fast_sq.cu: 32-bit Barrett, small moduli
struct FqState;        // ntt_fast_fq.cu: float-quotient products on the 8-coefficient schedule
struct Fq32State;      // ntt_fast_fq32.cu: float-quotient products on the warp-local schedule
struct Sh32State;      // ntt_fast_sh32.cu: Shoup products on the warp-local schedule, moduli up to 2^26
struct Xw32State;      // ntt_exact_w32.cu: variant-exact transforms on the warp-local schedule

// Device-resident state of one (q, n, variant) parameter set.  Zero-initialised by scgpu_ntt_plan_create; a state
// pointer is nullptr when its arithmetic does not apply to (q, n).
struct NttPlanDev {
    int n, logn, variant, tw_bits, device;
    RedConst rc;
    int32_t *w;          // caller's w[n], sign-extended to 32 bits
    int32_t *r;          // caller's r[n]
    int sm_count;
    int inputs_in_range;                 // SCGPU_PLAN_INPUTS_IN_RANGE: the fused products skip the range vote
    MontState *mont;
    SqState *sq;
    FqState *fq;
    Fq32State *fq32;
    Sh32State *sh32;
    Xw32State *xw32;
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
// e != nullptr (the *_add entry points): out = (product + e) mod q, e laid out like out and possibly out itself
int launch_polymul(const NttPlanDev &plan, int32_t *out, const int32_t *a, const int32_t *b,
                   size_t b_stride, size_t count, cudaStream_t stream, const int32_t *e = nullptr);
int launch_mul_key(const NttPlanDev &plan, int32_t *out, const int32_t *t, const void *key,
                   int key_bits, size_t key_stride, size_t count, cudaStream_t stream, const int32_t *e = nullptr);
// shared: A is ONE matrix [k][l][n] for all `count` instances (scgpu_matvec_shared_batch)
int launch_matvec(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s,
                  int k, int l, size_t count, cudaStream_t stream, bool shared = false, const int32_t *e = nullptr);
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
                        size_t b_stride, size_t count, cudaStream_t stream, const int32_t *e = nullptr);
int build_sh32_tables(NttPlanDev &plan, const int32_t *w_host);
void free_sh32_tables(NttPlanDev &plan);
int launch_polymul_sh32(const NttPlanDev &plan, int mode, int32_t *out, const int32_t *a, const void *b,
                        size_t b_stride, size_t count, cudaStream_t stream, const int32_t *e = nullptr);
int launch_matvec_sh32(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                       size_t count, cudaStream_t stream, bool shared = false, const int32_t *e = nullptr);
int launch_ntt_fq32(const NttPlanDev &plan, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_ntt_sh32(const NttPlanDev &plan, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_ntt_canonical(const NttPlanDev &plan, int inverse, int32_t *out, const int32_t *a, size_t count, cudaStream_t stream);
int launch_matvec_fq32(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                       size_t count, cudaStream_t stream, bool shared = false, const int32_t *e = nullptr);
// largest l of the mat-vec of a warp-local arithmetic the plan has (0: none)
int fq32_matvec_lmax(const NttPlanDev &plan);
int sh32_matvec_lmax(const NttPlanDev &plan);
int launch_matvec_fq(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                     size_t count, cudaStream_t stream, bool shared = false);
int build_sq_tables(NttPlanDev &plan, const int32_t *w_host);
void free_sq_tables(NttPlanDev &plan);
int launch_polymul_sq(const NttPlanDev &plan, int mode, int32_t *out, const int32_t *a, const void *b,
                      size_t b_stride, size_t count, cudaStream_t stream);
int launch_matvec_sq(const NttPlanDev &plan, int32_t *out, const int32_t *A, const int32_t *s, int k, int l,
                     size_t count, cudaStream_t stream, bool shared = false);

}  // namespace scgpu
