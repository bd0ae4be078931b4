// shim.cu -- the C-ABI of libscgpu.so: plans, batch entry points on device and host buffers,
// and the reference's drop-in NTT surface (utils_arith_ntt / init_reduce / barrett_init /
// roots_of_unity_s16/s32).  Host code only; every arithmetic result comes from a kernel in
// ntt_exact.cu / ntt_fast.cu.  There is no CPU evaluation path here.
#include "scgpu_internal.h"
#include "../../include/scgpu.h"
#include "../../include/scgpu_dropin.h"

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

namespace scgpu {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// Work counters of the persistent warp-local kernels (warp32.cuh: claim_next).  A ring of slots per device; a launch
// takes the next slot and zeroes it on its own stream, so launches in flight on different streams never share one
// (the ring is far longer than any queue of launches).  *ctr stays nullptr with SCGPU_STATIC_SCHED=1.
namespace {
constexpr int kCtrMaxDev = 64;
constexpr unsigned kCtrSlots = 8192;
std::mutex g_ctr_mu;
// A slot is 16 bytes: the 64-bit counter (cleared per launch; only its low word counts) and, written once when the
// ring is created, the number of groups one claim of that slot hands out (warp32.cuh: Claim).  Slot i serves the
// chunk size 1 << (i % 3), so a launcher picks its chunk size by picking the slot class -- no extra kernel argument.
constexpr unsigned kCtrClasses = 3;
constexpr unsigned kCtrPerClass = kCtrSlots / kCtrClasses;
unsigned long long *g_ctr_pool[kCtrMaxDev] = {};
unsigned g_ctr_next[kCtrMaxDev][kCtrClasses] = {};
}  // namespace

// Stream-ordered scratch (cudaMallocAsync: DRBG round keys, the L2-resident matrix chunk, staging of the *_host twins)
// comes from the device's default memory pool.  Its release threshold is 0 by default, i.e. every stream
// synchronisation hands the freed blocks back to the driver and the next call pays for real allocations again
// (measured: 75 ms instead of 12 ms per scgpu_gauss_streams_host call).  Keep up to 1 GiB cached.
int init_mempool()
{
    int dev = 0;
    SCGPU_CUDA_CHECK(cudaGetDevice(&dev));
    static std::atomic<uint64_t> done{0};
    if (dev >= 0 && dev < 64 && (done.load() >> dev) & 1) return SCGPU_OK;
    cudaMemPool_t pool;
    SCGPU_CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t cur = 0, want = 1ull << 30;
    SCGPU_CUDA_CHECK(cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &cur));
    if (cur < want) SCGPU_CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &want));
    if (dev >= 0 && dev < 64) done.fetch_or(1ull << dev);
    return SCGPU_OK;
}

// Allocates the current device's ring (called at plan creation, so that no launch ever allocates -- launches may be
// inside a stream capture).
int init_work_counters()
{
    int dev = 0;
    SCGPU_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kCtrMaxDev) return SCGPU_OK;
    std::lock_guard<std::mutex> lk(g_ctr_mu);
    if (!g_ctr_pool[dev]) {
        std::vector<unsigned> img((size_t)kCtrSlots * 4, 0u);
        for (unsigned i = 0; i < kCtrSlots; i++) img[(size_t)i * 4 + 2] = 1u << (i % kCtrClasses);
        unsigned long long *pool = nullptr;
        SCGPU_CUDA_CHECK(cudaMalloc(&pool, img.size() * sizeof(unsigned)));
        if (cudaMemcpy(pool, img.data(), img.size() * sizeof(unsigned), cudaMemcpyHostToDevice) != cudaSuccess) {
            cudaFree(pool);
            set_error("work counters: cudaMemcpy failed");
            return SCGPU_ERR_CUDA;
        }
        g_ctr_pool[dev] = pool;
    }
    return init_mempool();
}

int next_work_counter(cudaStream_t st, unsigned long long **ctr, int chunk)
{
    *ctr = nullptr;
    if (const char *ce = getenv("SCGPU_CLAIM_CHUNK")) { const int v = atoi(ce); if (v == 1 || v == 2 || v == 4) chunk = v; }
    const unsigned cls = chunk >= 4 ? 2u : chunk == 2 ? 1u : 0u;
    const char *env = getenv("SCGPU_STATIC_SCHED");
    if (env && atoi(env) != 0) return SCGPU_OK;
    // A captured graph would bake its slot into every replay, long after the ring has handed the slot to other
    // launches: captured launches keep the static stride.
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) { cudaGetLastError(); return SCGPU_OK; }
    int dev = 0;
    SCGPU_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kCtrMaxDev) return SCGPU_OK;
    unsigned long long *slot;
    {
        std::lock_guard<std::mutex> lk(g_ctr_mu);
        if (!g_ctr_pool[dev]) return SCGPU_OK;             // no plan was created on this device: static stride
        slot = g_ctr_pool[dev] + 2 * (size_t)((g_ctr_next[dev][cls]++ % kCtrPerClass) * kCtrClasses + cls);
    }
    SCGPU_CUDA_CHECK(cudaMemsetAsync(slot, 0, sizeof(unsigned long long), st));
    *ctr = slot;
    return SCGPU_OK;
}

}  // namespace scgpu

using namespace scgpu;

struct scgpu_ntt_plan {
    NttPlanDev dev;
    // staging for the *_host entry points (lazily created, guarded by mu)
    std::mutex mu;
    static constexpr int kStreams = 3;
    cudaStream_t streams[kStreams] = {nullptr, nullptr, nullptr};
    int32_t *d_a[kStreams] = {nullptr, nullptr, nullptr};
    int32_t *d_b[kStreams] = {nullptr, nullptr, nullptr};
    int32_t *d_o[kStreams] = {nullptr, nullptr, nullptr};
    int32_t *d_rc[kStreams] = {nullptr, nullptr, nullptr};
    void *d_shared = nullptr;      // a shared (b_stride == 0) second operand
    size_t shared_cap = 0;
    size_t staging_bytes = 0;      // capacity of each of d_a / d_b / d_o
    size_t staging_rc = 0;         // capacity of d_rc in rows
};

extern "C" const char *scgpu_last_error(void) { return g_err; }
extern "C" uint64_t scgpu_launch_count(void) { return g_launches.load(); }
extern "C" int scgpu_force_montgomery(int on) { return set_force_montgomery(on); }
extern "C" int scgpu_set_fast_arith(int mode) { return set_fast_arith(mode); }
extern "C" int scgpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

static int ilog2_exact(size_t n)
{
    int l = 0;
    while (((size_t)1 << l) < n) l++;
    return (((size_t)1 << l) == n) ? l : -1;
}

extern "C" int scgpu_ntt_plan_create(scgpu_ntt_plan_t **out, const void *params, int variant,
                                     const void *w, const void *r, int tw_bits, int device)
{
    if (!out || !params) { set_error("plan_create: null argument"); return SCGPU_ERR_ARG; }
    const ntt_params_t *p = static_cast<const ntt_params_t *>(params);
    if (variant < SCGPU_NTT_REFERENCE || variant > SCGPU_NTT_SOLINAS_8380417) {
        set_error("plan_create: reduction variant %d is not live in the reference (arith.c:360-396)", variant);
        return SCGPU_ERR_UNSUPPORTED;
    }
    if (tw_bits != 16 && tw_bits != 32 && !(tw_bits == 0 && !w)) { set_error("plan_create: tw_bits must be 16 or 32"); return SCGPU_ERR_ARG; }
    const int32_t q = p->u.ntt32.q;
    if (q < 2) { set_error("plan_create: q=%d", q); return SCGPU_ERR_ARG; }
    int ndev = 0;
    SCGPU_CUDA_CHECK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { set_error("plan_create: device %d of %d", device, ndev); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(device));

    struct Guard {                       // frees the plan on every early return below
        scgpu_ntt_plan *p;
        ~Guard() { if (p) scgpu_ntt_plan_destroy(p); }
    } guard{new scgpu_ntt_plan()};
    scgpu_ntt_plan *plan = guard.p;
    NttPlanDev &d = plan->dev;
    memset(&d, 0, sizeof(d));
    d.n = (int)p->n;
    d.logn = ilog2_exact(p->n);
    d.variant = variant;
    d.tw_bits = tw_bits;
    d.device = device;
    d.rc.q = q;
    d.rc.m = p->u.ntt32.m;
    d.rc.k = p->u.ntt32.k;
    d.rc.inv_q_dbl = p->inv_q_dbl;
    d.rc.qs_inv = (float)p->inv_q_dbl;
    d.rc.recip64 = ~0ull / (uint64_t)q;
    d.rc.recip32 = 0xFFFFFFFFu / (uint32_t)q;
    cudaDeviceProp prop;
    SCGPU_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    d.sm_count = prop.multiProcessorCount;
    { const int e = init_work_counters(); if (e != SCGPU_OK) return e; }
    if (w) {
        if (d.logn < 8 || d.logn > 10) {
            set_error("plan_create: transforms support n = 256, 512, 1024 (got %zu)", p->n);
            return SCGPU_ERR_UNSUPPORTED;
        }
        std::vector<int32_t> wh(d.n), rh(d.n);
        for (int i = 0; i < d.n; i++) {
            wh[i] = tw_bits == 16 ? (int32_t)static_cast<const int16_t *>(w)[i] : static_cast<const int32_t *>(w)[i];
            if (r) rh[i] = tw_bits == 16 ? (int32_t)static_cast<const int16_t *>(r)[i] : static_cast<const int32_t *>(r)[i];
        }
        SCGPU_CUDA_CHECK(cudaMalloc(&d.w, sizeof(int32_t) * d.n));
        SCGPU_CUDA_CHECK(cudaMemcpy(d.w, wh.data(), sizeof(int32_t) * d.n, cudaMemcpyHostToDevice));
        if (r) {
            SCGPU_CUDA_CHECK(cudaMalloc(&d.r, sizeof(int32_t) * d.n));
            SCGPU_CUDA_CHECK(cudaMemcpy(d.r, rh.data(), sizeof(int32_t) * d.n, cudaMemcpyHostToDevice));
        }
        int rcode = build_fast_tables(d, wh.data());
        if (rcode == SCGPU_OK) rcode = build_sq_tables(d, wh.data());
        if (rcode == SCGPU_OK) rcode = build_fq_tables(d, wh.data());
        if (rcode == SCGPU_OK) rcode = build_fq32_tables(d, wh.data());
        // needed where the float-quotient arithmetic does not apply; built for every modulus it can serve so that
        // scgpu_set_fast_arith(4) can cross-check it against the other arithmetics
        if (rcode == SCGPU_OK) rcode = build_sh32_tables(d, wh.data());
        if (rcode == SCGPU_OK) rcode = build_xw32_tables(d, wh.data(), r ? rh.data() : nullptr);
        if (rcode != SCGPU_OK) return rcode;
    }
    guard.p = nullptr;
    *out = plan;
    return SCGPU_OK;
}

extern "C" int scgpu_ntt_plan_set_flags(scgpu_ntt_plan_t *plan, unsigned flags)
{
    if (!plan || (flags & ~SCGPU_PLAN_INPUTS_IN_RANGE)) { set_error("plan_set_flags: bad argument"); return SCGPU_ERR_ARG; }
    const int prev = plan->dev.inputs_in_range ? (int)SCGPU_PLAN_INPUTS_IN_RANGE : 0;
    plan->dev.inputs_in_range = (flags & SCGPU_PLAN_INPUTS_IN_RANGE) ? 1 : 0;
    return prev;
}

extern "C" void scgpu_ntt_plan_destroy(scgpu_ntt_plan_t *plan)
{
    if (!plan) return;
    cudaSetDevice(plan->dev.device);
    for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) {
        if (plan->streams[i]) { cudaStreamSynchronize(plan->streams[i]); cudaStreamDestroy(plan->streams[i]); }
        cudaFree(plan->d_a[i]); cudaFree(plan->d_b[i]); cudaFree(plan->d_o[i]); cudaFree(plan->d_rc[i]);
    }
    cudaFree(plan->d_shared);
    cudaFree(plan->dev.w);
    cudaFree(plan->dev.r);
    free_fast_tables(plan->dev);
    free_sq_tables(plan->dev);
    free_fq_tables(plan->dev);
    free_fq32_tables(plan->dev);
    free_sh32_tables(plan->dev);
    free_xw32_tables(plan->dev);
    delete plan;
}

static bool op_needs_w(int op)
{
    return op <= SCGPU_OP_FFT_LARGE || op == SCGPU_OP_POLYMUL || op == SCGPU_OP_TRIPLE16;
}
static bool op_needs_r(int op)
{
    return op == SCGPU_OP_INV || op == SCGPU_OP_INV_LARGE || op == SCGPU_OP_POLYMUL || op == SCGPU_OP_TRIPLE16;
}
static bool op_needs_b(int op)
{
    return op == SCGPU_OP_PW || op == SCGPU_OP_PW16 || op == SCGPU_OP_POLYMUL || op == SCGPU_OP_TRIPLE16 ||
           op == SCGPU_OP_MULN || op == SCGPU_OP_DIV || op == SCGPU_OP_PWR || op == SCGPU_OP_SPARSE32 ||
           op == SCGPU_OP_SPARSE16;
}
static size_t b_elem_size(int op) { return (op == SCGPU_OP_PW16 || op == SCGPU_OP_TRIPLE16) ? 2 : 4; }
static size_t a_elem_size(int op) { return op == SCGPU_OP_SPARSE16 ? 2 : 4; }

static int check_batch_args(const scgpu_ntt_plan_t *plan, int op, const void *out, const void *a, const void *b)
{
    if (!plan || !out || !a) { set_error("ntt_batch: null argument"); return SCGPU_ERR_ARG; }
    if (op < 0 || op > SCGPU_OP_SPARSE16) { set_error("ntt_batch: unknown op %d", op); return SCGPU_ERR_ARG; }
    if (op_needs_w(op) && !plan->dev.w) { set_error("ntt_batch: op %d needs the plan's w table", op); return SCGPU_ERR_ARG; }
    if (op_needs_r(op) && !plan->dev.r) { set_error("ntt_batch: op %d needs the plan's r table", op); return SCGPU_ERR_ARG; }
    if (op_needs_b(op) && !b) { set_error("ntt_batch: op %d needs a second operand", op); return SCGPU_ERR_ARG; }
    if (op == SCGPU_OP_TRIPLE16 && plan->dev.tw_bits != 16) { set_error("TRIPLE16 needs 16-bit tables"); return SCGPU_ERR_ARG; }
    return SCGPU_OK;
}

extern "C" int scgpu_ntt_batch(const scgpu_ntt_plan_t *plan, int op, int32_t *out, const void *a,
                               const void *b, size_t b_stride, size_t count, int32_t scalar,
                               int32_t *rc, void *stream)
{
    int e = check_batch_args(plan, op, out, a, b);
    if (e != SCGPU_OK) return e;
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    ExactArgs g;
    g.out = out; g.a = a; g.b = op_needs_b(op) ? b : nullptr; g.b_stride = b_stride; g.count = count;
    g.w = plan->dev.w; g.r = plan->dev.r; g.rcodes = rc; g.rc = plan->dev.rc;
    g.op = op; g.tw_bits = plan->dev.tw_bits; g.scalar = scalar;
    return launch_exact(plan->dev, g, static_cast<cudaStream_t>(stream));
}

extern "C" int scgpu_polymul_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *a,
                                   const int32_t *b, size_t b_stride, size_t count, void *stream)
{
    if (!plan || !out || !a || !b) { set_error("polymul_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_polymul(plan->dev, out, a, b, b_stride, count, static_cast<cudaStream_t>(stream));
}

extern "C" int scgpu_ntt_canonical_batch(const scgpu_ntt_plan_t *plan, int inverse, int32_t *out, const int32_t *a,
                                         size_t count, void *stream)
{
    if (!plan || !out || !a) { set_error("ntt_canonical_batch: null argument"); return SCGPU_ERR_ARG; }
    if (!plan->dev.w || (inverse && !plan->dev.r)) { set_error("ntt_canonical_batch: the plan has no twiddle tables"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int e = launch_ntt_canonical(plan->dev, inverse, out, a, count, st);
    if (e != SCGPU_ERR_UNSUPPORTED) return e;
    // moduli outside both fused arithmetics: the variant-exact kernels compose the same result
    if (inverse) return scgpu_ntt_batch(plan, SCGPU_OP_INV, out, a, nullptr, 0, count, 0, nullptr, stream);
    const int e2 = scgpu_ntt_batch(plan, SCGPU_OP_FWD, out, a, nullptr, 0, count, 0, nullptr, stream);
    if (e2 != SCGPU_OK) return e2;
    return scgpu_ntt_batch(plan, SCGPU_OP_NORMALIZE, out, out, nullptr, 0, count, 0, nullptr, stream);
}

extern "C" int scgpu_ntt_mul_key_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *t,
                                       const void *key, int key_bits, size_t key_stride, size_t count,
                                       void *stream)
{
    if (!plan || !out || !t || !key) { set_error("ntt_mul_key_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_mul_key(plan->dev, out, t, key, key_bits, key_stride, count, static_cast<cudaStream_t>(stream));
}

extern "C" int scgpu_matvec_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *A,
                                  const int32_t *s, int k, int l, size_t count, void *stream)
{
    if (!plan || !out || !A || !s) { set_error("matvec_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_matvec(plan->dev, out, A, s, k, l, count, static_cast<cudaStream_t>(stream));
}

extern "C" int scgpu_matvec_shared_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *A,
                                         const int32_t *s, int k, int l, size_t count, void *stream)
{
    if (!plan || !out || !A || !s) { set_error("matvec_shared_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_matvec(plan->dev, out, A, s, k, l, count, static_cast<cudaStream_t>(stream), true);
}

// ---- the products above with an addend: out = (product + e) mod q ---------------------------------------------------

extern "C" int scgpu_polymul_add_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *a, const int32_t *b,
                                       size_t b_stride, const int32_t *e, size_t count, void *stream)
{
    if (!plan || !out || !a || !b || !e) { set_error("polymul_add_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_polymul(plan->dev, out, a, b, b_stride, count, static_cast<cudaStream_t>(stream), e);
}

extern "C" int scgpu_ntt_mul_key_add_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *t, const void *key,
                                           int key_bits, size_t key_stride, const int32_t *e, size_t count, void *stream)
{
    if (!plan || !out || !t || !key || !e) { set_error("ntt_mul_key_add_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_mul_key(plan->dev, out, t, key, key_bits, key_stride, count, static_cast<cudaStream_t>(stream), e);
}

extern "C" int scgpu_matvec_add_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *A, const int32_t *s,
                                      const int32_t *e, int k, int l, size_t count, void *stream)
{
    if (!plan || !out || !A || !s || !e) { set_error("matvec_add_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_matvec(plan->dev, out, A, s, k, l, count, static_cast<cudaStream_t>(stream), false, e);
}

extern "C" int scgpu_matvec_shared_add_batch(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *A, const int32_t *s,
                                             const int32_t *e, int k, int l, size_t count, void *stream)
{
    if (!plan || !out || !A || !s || !e) { set_error("matvec_shared_add_batch: null argument"); return SCGPU_ERR_ARG; }
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    return launch_matvec(plan->dev, out, A, s, k, l, count, static_cast<cudaStream_t>(stream), true, e);
}

// ---- module product with the matrix sampled on the device (rand_product.cu) ----------------------------------------

static int check_rand_args(const char *what, int prng_type, size_t seed_len, int n, int k, int l)
{
    if (prng_type != SCGPU_PRNG_AES_CTR_DRBG && prng_type != SCGPU_PRNG_CHACHA) {
        set_error("%s: PRNG type %d is not on the GPU path (0 = AES-CTR-DRBG, 2 = ChaCha20)", what, prng_type);
        return SCGPU_ERR_UNSUPPORTED;
    }
    if (seed_len == 0 || k < 1 || l < 1) { set_error("%s: bad shape (k=%d l=%d)", what, k, l); return SCGPU_ERR_ARG; }
    if (n != 256) {
        // uniform_random_ring_q_csprng (module_lwe.c:519-535) never advances its output pointer: for n > 256 every
        // 256-coefficient block lands on a[0..255] and the rest of the ring keeps whatever the caller's buffer held.
        // Kyber and Dilithium are n = 256; nothing else has a defined result.
        set_error("%s: the reference's ring sampler is only defined for n = 256 (got %d)", what, n);
        return SCGPU_ERR_UNSUPPORTED;
    }
    if ((size_t)k * l * n * 2 >= 0x01000000u) { set_error("%s: an instance would cross the generator's 16 MiB reseed period", what); return SCGPU_ERR_UNSUPPORTED; }
    return SCGPU_OK;
}

extern "C" int scgpu_rand_matrix_csprng_batch(int32_t *A, const uint8_t *seeds, size_t seed_len, int prng_type, int32_t q,
                                              uint32_t q_bits, int n, int k, int l, int transpose, size_t count, void *stream)
{
    if (!A || !seeds) { set_error("rand_matrix: null argument"); return SCGPU_ERR_ARG; }
    // the generation kernels store whole 8- and 16-byte groups of coefficients (a ring is 1 KiB, so every ring of an
    // aligned A is aligned too)
    if (reinterpret_cast<uintptr_t>(A) % 16 != 0) { set_error("rand_matrix: A is not 16-byte aligned"); return SCGPU_ERR_ARG; }
    const int e = check_rand_args("rand_matrix", prng_type, seed_len, n, k, l);
    if (e != SCGPU_OK) return e;
    return launch_gen_rings(prng_type, seeds, seed_len, count, A, n, k, l, transpose, q, q_bits, static_cast<cudaStream_t>(stream));
}

extern "C" int scgpu_rand_product_csprng_batch(const scgpu_ntt_plan_t *plan, int32_t *t, const int32_t *y, const uint8_t *seeds,
                                               size_t seed_len, int prng_type, uint32_t q_bits, int k, int l, int transpose,
                                               size_t count, void *stream)
{
    if (!plan || !t || !y || !seeds) { set_error("rand_product: null argument"); return SCGPU_ERR_ARG; }
    if (!plan->dev.w || !plan->dev.r) { set_error("rand_product: the plan has no twiddle tables"); return SCGPU_ERR_ARG; }
    const int n = plan->dev.n;
    int e = check_rand_args("rand_product", prng_type, seed_len, n, k, l);
    if (e != SCGPU_OK) return e;
    if (transpose && plan->dev.tw_bits == 32 && l > 1) {
        set_error("rand_product: create_rand_product_32_csprng's transposed branch adds the matrix ring instead of the running sum "
                  "(module_lwe.c:623-628); no scheme calls it and it is not reproduced");
        return SCGPU_ERR_UNSUPPORTED;
    }
    if (count == 0) return SCGPU_OK;
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the matrix of a chunk of instances stays in the L2: 48 MB of the 126 MB
    const size_t inst_bytes = (size_t)k * l * n * sizeof(int32_t);
    size_t chunk = (48u << 20) / inst_bytes;
    if (chunk < 1) chunk = 1;
    if (chunk > count) chunk = count;
    int32_t *scratch = nullptr;
    SCGPU_CUDA_CHECK(cudaMallocAsync(&scratch, chunk * inst_bytes, st));
    for (size_t off = 0; off < count && e == SCGPU_OK; off += chunk) {
        const size_t cnt = count - off < chunk ? count - off : chunk;
        e = launch_gen_rings(prng_type, seeds + off * seed_len, seed_len, cnt, scratch, n, k, l, transpose, plan->dev.rc.q, q_bits, st);
        if (e == SCGPU_OK) e = launch_matvec(plan->dev, t + off * (size_t)k * n, scratch, y + off * (size_t)l * n, k, l, cnt, st);
    }
    SCGPU_CUDA_CHECK(cudaFreeAsync(scratch, st));
    return e;
}

extern "C" int scgpu_rand_product_csprng_shared_batch(const scgpu_ntt_plan_t *plan, int32_t *t, const int32_t *y, const uint8_t *seed,
                                                      size_t seed_len, int prng_type, uint32_t q_bits, int k, int l, int transpose,
                                                      size_t count, void *stream)
{
    if (!plan || !t || !y || !seed) { set_error("rand_product_shared: null argument"); return SCGPU_ERR_ARG; }
    if (!plan->dev.w || !plan->dev.r) { set_error("rand_product_shared: the plan has no twiddle tables"); return SCGPU_ERR_ARG; }
    const int n = plan->dev.n;
    int e = check_rand_args("rand_product_shared", prng_type, seed_len, n, k, l);
    if (e != SCGPU_OK) return e;
    if (transpose && plan->dev.tw_bits == 32 && l > 1) {
        set_error("rand_product_shared: create_rand_product_32_csprng's transposed branch adds the matrix ring instead of the running "
                  "sum (module_lwe.c:623-628); no scheme calls it and it is not reproduced");
        return SCGPU_ERR_UNSUPPORTED;
    }
    if (count == 0) return SCGPU_OK;
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // one seed: the matrix is drawn once, then the whole batch runs the shared-matrix product (no chunking)
    int32_t *scratch = nullptr;
    SCGPU_CUDA_CHECK(cudaMallocAsync(&scratch, (size_t)k * l * n * sizeof(int32_t), st));
    e = launch_gen_rings(prng_type, seed, seed_len, 1, scratch, n, k, l, transpose, plan->dev.rc.q, q_bits, st);
    if (e == SCGPU_OK) e = launch_matvec(plan->dev, t, scratch, y, k, l, count, st, true);
    SCGPU_CUDA_CHECK(cudaFreeAsync(scratch, st));
    return e;
}

// three-stream pipeline over chunks of instances: y (and the seeds) in, t out; the matrix never crosses the bus.
// shared: ONE seed for every instance, copied once
static int rand_product_host(const scgpu_ntt_plan_t *plan, int32_t *t, const int32_t *y, const uint8_t *seeds, size_t seed_len,
                             int prng_type, uint32_t q_bits, int k, int l, int transpose, size_t count, bool shared)
{
    // before the pipeline is sized from k and l (k = l = 0 would divide by zero below)
    const int e0 = check_rand_args(shared ? "rand_product_shared_host" : "rand_product_host", prng_type, seed_len, plan->dev.n, k, l);
    if (e0 != SCGPU_OK) return e0;
    if (count == 0) return SCGPU_OK;
    scgpu_ntt_plan *p = const_cast<scgpu_ntt_plan *>(plan);
    std::lock_guard<std::mutex> lock(p->mu);
    SCGPU_CUDA_CHECK(cudaSetDevice(p->dev.device));
    for (int i = 0; i < scgpu_ntt_plan::kStreams; i++)
        if (!p->streams[i]) SCGPU_CUDA_CHECK(cudaStreamCreateWithFlags(&p->streams[i], cudaStreamNonBlocking));
    // three-stream pipeline over chunks of instances: seeds + y in, t out; the matrix never crosses the bus
    const size_t n = (size_t)p->dev.n;
    const size_t yb = (size_t)l * n * 4, tb = (size_t)k * n * 4;
    size_t rows = (16u << 20) / (yb > tb ? yb : tb);
    if (rows < 1) rows = 1;
    if (rows > count) rows = count;
    int status = SCGPU_OK;
    void *dy[scgpu_ntt_plan::kStreams] = {}, *dt[scgpu_ntt_plan::kStreams] = {}, *ds[scgpu_ntt_plan::kStreams] = {};
    void *dseed = nullptr;                                   // shared: the one seed, read by every stream
    auto cuda_ok = [&](cudaError_t e, const char *what) {
        if (e != cudaSuccess && status == SCGPU_OK) { set_error("%s failed: %s", what, cudaGetErrorString(e)); status = SCGPU_ERR_CUDA; }
        return e == cudaSuccess;
    };
    if (shared && cuda_ok(cudaMallocAsync(&dseed, seed_len, p->streams[0]), "cudaMallocAsync")
        && cuda_ok(cudaMemcpyAsync(dseed, seeds, seed_len, cudaMemcpyHostToDevice, p->streams[0]), "H2D copy"))
        cuda_ok(cudaStreamSynchronize(p->streams[0]), "cudaStreamSynchronize");
    for (int i = 0; i < scgpu_ntt_plan::kStreams && status == SCGPU_OK; i++) {
        cuda_ok(cudaMallocAsync(&dy[i], rows * yb, p->streams[i]), "cudaMallocAsync");
        cuda_ok(cudaMallocAsync(&dt[i], rows * tb, p->streams[i]), "cudaMallocAsync");
        if (!shared) cuda_ok(cudaMallocAsync(&ds[i], rows * seed_len, p->streams[i]), "cudaMallocAsync");
    }
    for (size_t off = 0, ci = 0; off < count && status == SCGPU_OK; off += rows, ci++) {
        const int s = (int)(ci % scgpu_ntt_plan::kStreams);
        cudaStream_t st = p->streams[s];
        const size_t cnt = count - off < rows ? count - off : rows;
        if (!cuda_ok(cudaMemcpyAsync(dy[s], reinterpret_cast<const char *>(y) + off * yb, cnt * yb, cudaMemcpyHostToDevice, st), "H2D copy")) break;
        int e;
        if (shared) {
            e = scgpu_rand_product_csprng_shared_batch(plan, static_cast<int32_t *>(dt[s]), static_cast<const int32_t *>(dy[s]),
                                                       static_cast<const uint8_t *>(dseed), seed_len, prng_type, q_bits, k, l, transpose, cnt, st);
        } else {
            if (!cuda_ok(cudaMemcpyAsync(ds[s], seeds + off * seed_len, cnt * seed_len, cudaMemcpyHostToDevice, st), "H2D copy")) break;
            e = scgpu_rand_product_csprng_batch(plan, static_cast<int32_t *>(dt[s]), static_cast<const int32_t *>(dy[s]),
                                                static_cast<const uint8_t *>(ds[s]), seed_len, prng_type, q_bits, k, l, transpose, cnt, st);
        }
        if (e != SCGPU_OK) { status = e; break; }
        cuda_ok(cudaMemcpyAsync(reinterpret_cast<char *>(t) + off * tb, dt[s], cnt * tb, cudaMemcpyDeviceToHost, st), "D2H copy");
    }
    // every path releases the staging buffers and drains the streams
    for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) {
        if (dy[i]) cudaFreeAsync(dy[i], p->streams[i]);
        if (dt[i]) cudaFreeAsync(dt[i], p->streams[i]);
        if (ds[i]) cudaFreeAsync(ds[i], p->streams[i]);
        cuda_ok(cudaStreamSynchronize(p->streams[i]), "cudaStreamSynchronize");
    }
    if (dseed) {                                             // every stream has drained: nobody reads the seed any more
        cudaFreeAsync(dseed, p->streams[0]);
        cuda_ok(cudaStreamSynchronize(p->streams[0]), "cudaStreamSynchronize");
    }
    return status;
}

extern "C" int scgpu_rand_product_csprng_batch_host(const scgpu_ntt_plan_t *plan, int32_t *t, const int32_t *y, const uint8_t *seeds,
                                                    size_t seed_len, int prng_type, uint32_t q_bits, int k, int l, int transpose,
                                                    size_t count)
{
    if (!plan || !t || !y || !seeds) { set_error("rand_product_host: null argument"); return SCGPU_ERR_ARG; }
    return rand_product_host(plan, t, y, seeds, seed_len, prng_type, q_bits, k, l, transpose, count, false);
}

extern "C" int scgpu_rand_product_csprng_shared_batch_host(const scgpu_ntt_plan_t *plan, int32_t *t, const int32_t *y,
                                                           const uint8_t *seed, size_t seed_len, int prng_type, uint32_t q_bits,
                                                           int k, int l, int transpose, size_t count)
{
    if (!plan || !t || !y || !seed) { set_error("rand_product_shared_host: null argument"); return SCGPU_ERR_ARG; }
    return rand_product_host(plan, t, y, seed, seed_len, prng_type, q_bits, k, l, transpose, count, true);
}

// ---- host-buffer entry points: chunked three-stream pipeline -----------------------------------------

// Sizes the three staging buffers for THIS call and returns its chunk length in rows.  A chunk is a whole number of
// waves of the persistent fused kernels (sm_count x 20 one-warp CTAs x 1024/n rows per warp) so that no chunk ends on a
// partly filled wave, about 24 MiB of the widest operand: large enough to amortise the launch, small enough that H2D,
// kernel and D2H of neighbouring chunks overlap.
static int ensure_staging(scgpu_ntt_plan *plan, size_t row_bytes_a, size_t row_bytes_b, size_t row_bytes_o, size_t count,
                          size_t *chunk_rows)
{
    size_t widest = row_bytes_a > row_bytes_o ? row_bytes_a : row_bytes_o;
    if (row_bytes_b > widest) widest = row_bytes_b;
    if (widest == 0) widest = 4;
    size_t rows = (24u << 20) / widest;
    const size_t n = (size_t)plan->dev.n;
    const size_t wave = (size_t)(plan->dev.sm_count > 0 ? plan->dev.sm_count : 148) * 20 * (n && n <= 1024 ? 1024 / n : 1);
    if (rows > wave) rows -= rows % wave;
    if (rows < 1) rows = 1;
    if (rows > count) rows = count;
    const size_t need = rows * widest;
    for (int i = 0; i < scgpu_ntt_plan::kStreams; i++)
        if (!plan->streams[i]) SCGPU_CUDA_CHECK(cudaStreamCreateWithFlags(&plan->streams[i], cudaStreamNonBlocking));
    if (plan->staging_bytes < need) {
        for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) {
            SCGPU_CUDA_CHECK(cudaStreamSynchronize(plan->streams[i]));
            cudaFree(plan->d_a[i]); cudaFree(plan->d_b[i]); cudaFree(plan->d_o[i]);
            plan->d_a[i] = plan->d_b[i] = plan->d_o[i] = nullptr;
        }
        plan->staging_bytes = 0;
        for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) {
            SCGPU_CUDA_CHECK(cudaMalloc(&plan->d_a[i], need));
            SCGPU_CUDA_CHECK(cudaMalloc(&plan->d_b[i], need));
            SCGPU_CUDA_CHECK(cudaMalloc(&plan->d_o[i], need));
        }
        plan->staging_bytes = need;
    }
    if (plan->staging_rc < rows) {
        for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) {
            cudaFree(plan->d_rc[i]);
            plan->d_rc[i] = nullptr;
        }
        plan->staging_rc = 0;
        for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) SCGPU_CUDA_CHECK(cudaMalloc(&plan->d_rc[i], rows * sizeof(int32_t)));
        plan->staging_rc = rows;
    }
    *chunk_rows = rows;
    return SCGPU_OK;
}

static int ensure_shared(scgpu_ntt_plan *plan, const void *host, size_t bytes)
{
    if (plan->shared_cap < bytes) {
        cudaFree(plan->d_shared);
        plan->d_shared = nullptr;
        SCGPU_CUDA_CHECK(cudaMalloc(&plan->d_shared, bytes));
        plan->shared_cap = bytes;
    }
    SCGPU_CUDA_CHECK(cudaMemcpy(plan->d_shared, host, bytes, cudaMemcpyHostToDevice));
    return SCGPU_OK;
}

// kind: 0 exact op, 1 fused polymul, 2 fused key product (key_bits in `op`), 3 canonical transform (inverse in `op`)
static int run_host_pipeline(scgpu_ntt_plan *plan, int kind, int op, int32_t *out, const void *a, const void *b,
                             size_t b_stride, size_t count, int32_t scalar, int32_t *rc)
{
    if (count == 0) return SCGPU_OK;
    std::lock_guard<std::mutex> lock(plan->mu);
    SCGPU_CUDA_CHECK(cudaSetDevice(plan->dev.device));
    const size_t n = (size_t)plan->dev.n;
    const size_t ra = n * (kind == 0 ? a_elem_size(op) : 4);
    const size_t belem = kind == 0 ? b_elem_size(op) : (kind == 2 ? (size_t)op / 8 : 4);
    const bool has_b = kind == 3 ? false : (kind != 0 || op_needs_b(op));
    const size_t rb = has_b ? (b_stride ? b_stride : n) * belem : 0;
    size_t rows = 0;
    int e = ensure_staging(plan, ra, b_stride ? rb : 0, n * 4, count, &rows);
    if (e != SCGPU_OK) return e;
    const void *d_bshared = nullptr;
    if (has_b && b_stride == 0) {
        size_t bytes = (kind == 0 && (op == SCGPU_OP_SPARSE32 || op == SCGPU_OP_SPARSE16)) ? (size_t)(scalar & 0xFFFF) * 4 : n * belem;
        e = ensure_shared(plan, b, bytes);
        if (e != SCGPU_OK) return e;
        d_bshared = plan->d_shared;
    }
    int status = SCGPU_OK;
    for (size_t off = 0, ci = 0; off < count; off += rows, ci++) {
        const int s = (int)(ci % scgpu_ntt_plan::kStreams);
        cudaStream_t st = plan->streams[s];
        const size_t cnt = (count - off < rows) ? count - off : rows;
        SCGPU_CUDA_CHECK(cudaMemcpyAsync(plan->d_a[s], static_cast<const char *>(a) + off * ra, cnt * ra, cudaMemcpyHostToDevice, st));
        const void *db = d_bshared;
        if (has_b && b_stride) {
            SCGPU_CUDA_CHECK(cudaMemcpyAsync(plan->d_b[s], static_cast<const char *>(b) + off * rb, cnt * rb, cudaMemcpyHostToDevice, st));
            db = plan->d_b[s];
        }
        if (kind == 0) {
            ExactArgs g;
            g.out = plan->d_o[s]; g.a = plan->d_a[s]; g.b = has_b ? db : nullptr; g.b_stride = b_stride; g.count = cnt;
            g.w = plan->dev.w; g.r = plan->dev.r; g.rcodes = rc ? plan->d_rc[s] : nullptr; g.rc = plan->dev.rc;
            g.op = op; g.tw_bits = plan->dev.tw_bits; g.scalar = scalar;
            status = launch_exact(plan->dev, g, st);
        } else if (kind == 1) {
            status = launch_polymul(plan->dev, plan->d_o[s], plan->d_a[s], static_cast<const int32_t *>(db), b_stride, cnt, st);
        } else if (kind == 3) {
            status = scgpu_ntt_canonical_batch(plan, op, plan->d_o[s], plan->d_a[s], cnt, st);
        } else {
            status = launch_mul_key(plan->dev, plan->d_o[s], plan->d_a[s], db, op, b_stride, cnt, st);
        }
        if (status != SCGPU_OK) break;
        SCGPU_CUDA_CHECK(cudaMemcpyAsync(out + off * n, plan->d_o[s], cnt * n * 4, cudaMemcpyDeviceToHost, st));
        if (rc && kind == 0) SCGPU_CUDA_CHECK(cudaMemcpyAsync(rc + off, plan->d_rc[s], cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    for (int i = 0; i < scgpu_ntt_plan::kStreams; i++) SCGPU_CUDA_CHECK(cudaStreamSynchronize(plan->streams[i]));
    return status;
}

extern "C" int scgpu_ntt_batch_host(const scgpu_ntt_plan_t *plan, int op, int32_t *out, const void *a,
                                    const void *b, size_t b_stride, size_t count, int32_t scalar, int32_t *rc)
{
    int e = check_batch_args(plan, op, out, a, b);
    if (e != SCGPU_OK) return e;
    return run_host_pipeline(const_cast<scgpu_ntt_plan *>(plan), 0, op, out, a, b, b_stride, count, scalar, rc);
}

extern "C" int scgpu_polymul_batch_host(const scgpu_ntt_plan_t *plan, int32_t *out, const int32_t *a,
                                        const int32_t *b, size_t b_stride, size_t count)
{
    if (!plan || !out || !a || !b) { set_error("polymul_batch_host: null argument"); return SCGPU_ERR_ARG; }
    return run_host_pipeline(const_cast<scgpu_ntt_plan *>(plan), 1, 0, out, a, b, b_stride, count, 0, nullptr);
}

extern "C" int scgpu_ntt_canonical_batch_host(const scgpu_ntt_plan_t *plan, int inverse, int32_t *out, const int32_t *a,
                                              size_t count)
{
    if (!plan || !out || !a) { set_error("ntt_canonical_batch_host: null argument"); return SCGPU_ERR_ARG; }
    return run_host_pipeline(const_cast<scgpu_ntt_plan *>(plan), 3, inverse ? 1 : 0, out, a, nullptr, 0, count, 0, nullptr);
}

// ---- one host batch over several devices (host-side scatter / gather, one thread per device) ---------------------

extern "C" int scgpu_ntt_plans_create_all(scgpu_ntt_plan_t **plans, int max_plans, const void *params, int variant,
                                          const void *w, const void *r, int tw_bits)
{
    if (!plans || max_plans < 1) { set_error("plans_create_all: null argument"); return SCGPU_ERR_ARG; }
    int ndev = scgpu_device_count();
    if (ndev < 1) { set_error("plans_create_all: no CUDA device"); return SCGPU_ERR_CUDA; }
    if (ndev > max_plans) ndev = max_plans;
    for (int d = 0; d < ndev; d++) {
        const int e = scgpu_ntt_plan_create(&plans[d], params, variant, w, r, tw_bits, d);
        if (e != SCGPU_OK) {
            for (int i = 0; i < d; i++) { scgpu_ntt_plan_destroy(plans[i]); plans[i] = nullptr; }
            return e;
        }
    }
    return ndev;
}

template <class Fn>
static int run_slabs(int nplans, size_t count, Fn fn)
{
    std::vector<std::thread> th;
    std::vector<int> status((size_t)nplans, SCGPU_OK);
    std::vector<std::string> msg((size_t)nplans);
    for (int i = 0; i < nplans; i++) {
        const size_t lo = count * (size_t)i / (size_t)nplans, hi = count * (size_t)(i + 1) / (size_t)nplans;
        if (hi == lo) continue;
        th.emplace_back([&, i, lo, hi] {
            status[i] = fn(i, lo, hi - lo);
            if (status[i] != SCGPU_OK) msg[i] = scgpu_last_error();          // the error text is per thread
        });
    }
    for (auto &t : th) t.join();
    for (int i = 0; i < nplans; i++)
        if (status[i] != SCGPU_OK) { set_error("device slab %d: %s", i, msg[i].c_str()); return status[i]; }
    return SCGPU_OK;
}

extern "C" int scgpu_polymul_batch_host_multi(const scgpu_ntt_plan_t *const *plans, int nplans, int32_t *out, const int32_t *a,
                                              const int32_t *b, size_t b_stride, size_t count)
{
    if (!plans || nplans < 1 || !out || !a || !b) { set_error("polymul_batch_host_multi: null argument"); return SCGPU_ERR_ARG; }
    for (int i = 0; i < nplans; i++) if (!plans[i]) { set_error("polymul_batch_host_multi: plan %d is null", i); return SCGPU_ERR_ARG; }
    const size_t n = (size_t)plans[0]->dev.n;
    return run_slabs(nplans, count, [&](int i, size_t lo, size_t cnt) {
        return scgpu_polymul_batch_host(plans[i], out + lo * n, a + lo * n, b + lo * b_stride, b_stride, cnt);
    });
}

extern "C" int scgpu_ntt_batch_host_multi(const scgpu_ntt_plan_t *const *plans, int nplans, int op, int32_t *out, const void *a,
                                          const void *b, size_t b_stride, size_t count, int32_t scalar, int32_t *rc)
{
    if (!plans || nplans < 1 || !out || !a) { set_error("ntt_batch_host_multi: null argument"); return SCGPU_ERR_ARG; }
    for (int i = 0; i < nplans; i++) if (!plans[i]) { set_error("ntt_batch_host_multi: plan %d is null", i); return SCGPU_ERR_ARG; }
    if (op < 0 || op > SCGPU_OP_SPARSE16) { set_error("ntt_batch_host_multi: unknown op %d", op); return SCGPU_ERR_ARG; }
    const size_t n = (size_t)plans[0]->dev.n;
    const size_t ea = a_elem_size(op), eb = b_elem_size(op);
    return run_slabs(nplans, count, [&](int i, size_t lo, size_t cnt) {
        const char *bp = b ? static_cast<const char *>(b) + lo * b_stride * eb : nullptr;
        return scgpu_ntt_batch_host(plans[i], op, out + lo * n, static_cast<const char *>(a) + lo * n * ea, bp, b_stride, cnt, scalar,
                                    rc ? rc + lo : nullptr);
    });
}

// =======================================================================================================
// Drop-in surface: utils_arith_ntt() and friends
// =======================================================================================================

extern "C" void barrett_init(ntt_params_t *p)
{
    // ntt.c:142-146
    p->u.ntt32.k = 30;
    p->u.ntt32.m = (1 << p->u.ntt32.k) / p->u.ntt32.q;
}

extern "C" void init_reduce(ntt_params_t *p, size_t n, SINT32 q)
{
    // ntt.c:132-140
    p->n = n;
    p->u.ntt32.q = q;
    barrett_init(p);
    p->q_dbl = (DOUBLE)q;
    p->inv_q_dbl = 1.0 / p->q_dbl;
    p->inv_q_flt = 1.0 / (FLOAT)q;
}

// roots_of_unity.c:141-207.  Table generation is host-side set-up (the reference does it at build
// time with build_tools/ntt_table_gen or once per create() under USE_RUNTIME_NTT_TABLES).
static uint64_t mulmod_u64(uint64_t a, uint64_t b, uint64_t q) { return (uint64_t)(((unsigned __int128)a * b) % q); }
static uint64_t powmod_u64(uint64_t b, uint64_t e, uint64_t q)
{
    uint64_t r = 1;
    b %= q;
    while (e) { if (e & 1) r = mulmod_u64(r, b, q); b = mulmod_u64(b, b, q); e >>= 1; }
    return r;
}
template <typename T>
static SINT32 roots_of_unity_impl(T *fwd, T *inv, size_t n, uint64_t p, uint64_t prim)
{
    if (prim == 0) {
        for (uint64_t m = 2; m + 1 < p; m++)
            if (powmod_u64(m, n, p) == p - 1) { prim = m; break; }       // smallest m with m^n == -1
    }
    if (prim == 0) return SC_FUNC_FAILURE;
    // inv[0] = |x| where n x + p y = 1; for the parameter sets of the reference this is -(n^-1) mod p
    uint64_t ninv = powmod_u64(n % p, p - 2, p);
    uint64_t acc = 1, racc = (p - ninv) % p;
    for (size_t i = 0; i < n; i++) {
        fwd[i] = (T)acc;
        inv[i] = (T)racc;
        acc = mulmod_u64(acc, prim, p);
        racc = mulmod_u64(racc, prim, p);
    }
    return SC_FUNC_SUCCESS;
}
extern "C" SINT32 roots_of_unity_s32(SINT32 *fwd, SINT32 *inv, size_t n, sc_ulimb_t p, sc_ulimb_t prim, SINT32 ternary)
{
    (void)ternary;
    return roots_of_unity_impl<SINT32>(fwd, inv, n, p, prim);
}
extern "C" SINT32 roots_of_unity_s16(SINT16 *fwd, SINT16 *inv, size_t n, sc_ulimb_t p, sc_ulimb_t prim, SINT32 ternary)
{
    (void)ternary;
    return roots_of_unity_impl<SINT16>(fwd, inv, n, p, prim);
}

namespace {

[[noreturn]] void dropin_fatal(const char *what)
{
    // The reference has no error channel on these void functions (SURVEY.md 8b): log and abort.
    fprintf(stderr, "libscgpu: %s: %s\n", what, scgpu_last_error());
    abort();
}

uint64_t fnv1a(const void *data, size_t bytes, uint64_t h = 1469598103934665603ull)
{
    const unsigned char *p = static_cast<const unsigned char *>(data);
    for (size_t i = 0; i < bytes; i++) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

// Plans of the drop-in calls.  A call is matched by its parameter VALUES and the ADDRESSES of its tables (a handful
// of words compared, no table is read); only an address that was not seen before has its table contents hashed, so
// that tables malloc'ed at run time (USE_RUNTIME_NTT_TABLES, bliss_b.c:365-374) and freed / re-created elsewhere
// find the plan that already holds the same contents.  Every hit also compares four sentinel twiddles kept with the
// entry, which catches an address re-used for different contents, and compares the full key, so neither a hash
// collision nor padding bytes can select a plan of another modulus.
struct PlanKey {
    const void *w, *r;
    uint64_t n;
    double inv;
    int32_t q, m, k;
    int variant, tw_bits, device;
    bool operator==(const PlanKey &o) const
    {
        return w == o.w && r == o.r && n == o.n && memcmp(&inv, &o.inv, sizeof(inv)) == 0 && q == o.q && m == o.m &&
               k == o.k && variant == o.variant && tw_bits == o.tw_bits && device == o.device;
    }
};
struct PlanKeyHash {
    size_t operator()(const PlanKey &k) const
    {
        uint64_t h = fnv1a(&k.w, sizeof(k.w));
        h = fnv1a(&k.r, sizeof(k.r), h); h = fnv1a(&k.n, sizeof(k.n), h); h = fnv1a(&k.inv, sizeof(k.inv), h);
        h = fnv1a(&k.q, sizeof(k.q), h); h = fnv1a(&k.m, sizeof(k.m), h); h = fnv1a(&k.k, sizeof(k.k), h);
        h = fnv1a(&k.variant, sizeof(k.variant), h); h = fnv1a(&k.tw_bits, sizeof(k.tw_bits), h);
        return (size_t)fnv1a(&k.device, sizeof(k.device), h);
    }
};
struct PlanEntry {
    scgpu_ntt_plan *plan = nullptr;
    int32_t sentinel[4] = {0, 0, 0, 0};        // w[1], w[n-1], r[1], r[n-1]
};

static void read_sentinels(const PlanKey &k, int32_t out[4])
{
    auto at = [&](const void *t, size_t i) -> int32_t {
        if (!t || i >= k.n) return 0;
        return k.tw_bits == 16 ? (int32_t)static_cast<const int16_t *>(t)[i] : static_cast<const int32_t *>(t)[i];
    };
    out[0] = at(k.w, 1); out[1] = at(k.w, (size_t)k.n - 1); out[2] = at(k.r, 1); out[3] = at(k.r, (size_t)k.n - 1);
}

struct PlanCache {
    std::mutex mu;
    std::unordered_map<PlanKey, PlanEntry, PlanKeyHash> by_addr;
    struct Content { PlanKey key; std::vector<unsigned char> w, r; scgpu_ntt_plan *plan; };
    std::unordered_multimap<uint64_t, Content> by_content;      // hash -> candidates, compared in full
    ~PlanCache()
    {
        // process exit: the CUDA context may already be gone; the driver reclaims device memory
    }
    scgpu_ntt_plan *get(const PlanKey &key)
    {
        int32_t sent[4];
        read_sentinels(key, sent);
        std::lock_guard<std::mutex> lock(mu);
        auto it = by_addr.find(key);
        if (it != by_addr.end() && memcmp(it->second.sentinel, sent, sizeof(sent)) == 0) return it->second.plan;
        // unknown address (or an address re-used for other contents): identify the tables by value
        const size_t tb = (size_t)(key.tw_bits / 8) * (size_t)key.n;
        PlanKey vkey = key;
        vkey.w = vkey.r = nullptr;
        uint64_t h = PlanKeyHash()(vkey);
        if (key.w) h = fnv1a(key.w, tb, h);
        if (key.r) h = fnv1a(key.r, tb, h ^ 0x9E3779B97F4A7C15ull);
        scgpu_ntt_plan *plan = nullptr;
        auto range = by_content.equal_range(h);
        for (auto c = range.first; c != range.second; ++c) {
            const Content &e = c->second;
            if (e.key == vkey && e.w.size() == (key.w ? tb : 0) && e.r.size() == (key.r ? tb : 0) &&
                (!key.w || memcmp(e.w.data(), key.w, tb) == 0) && (!key.r || memcmp(e.r.data(), key.r, tb) == 0)) {
                plan = e.plan;
                break;
            }
        }
        if (!plan) {
            ntt_params_t q;
            memset(&q, 0, sizeof(q));
            q.n = (size_t)key.n;
            q.u.ntt32.q = key.q; q.u.ntt32.m = key.m; q.u.ntt32.k = key.k;
            q.inv_q_dbl = key.inv; q.q_dbl = (double)key.q; q.inv_q_flt = (float)key.inv;
            if (scgpu_ntt_plan_create(&plan, &q, key.variant, key.w, key.r, key.w ? key.tw_bits : 0, key.device) != SCGPU_OK)
                dropin_fatal("plan creation failed");
            Content e;
            e.key = vkey; e.plan = plan;
            if (key.w) e.w.assign(static_cast<const unsigned char *>(key.w), static_cast<const unsigned char *>(key.w) + tb);
            if (key.r) e.r.assign(static_cast<const unsigned char *>(key.r), static_cast<const unsigned char *>(key.r) + tb);
            by_content.emplace(h, std::move(e));
        }
        PlanEntry pe;
        pe.plan = plan;
        memcpy(pe.sentinel, sent, sizeof(sent));
        by_addr[key] = pe;
        return plan;
    }
};
PlanCache g_cache;

int dropin_device()
{
    static const int dev = [] { const char *env = getenv("SCGPU_DEVICE"); return env ? atoi(env) : 0; }();
    return dev;
}

// Per-thread stream, scratch and last plan: the reference's functions are re-entrant and BLISS-B calls them from
// worker threads (bliss_b.c:74-175).  Released when the thread exits.
struct ThreadCtx {
    cudaStream_t st = nullptr;
    char *d[3] = {nullptr, nullptr, nullptr};
    size_t cap[3] = {0, 0, 0};
    int32_t *d_rc = nullptr;
    // Small calls go through one pinned, device-mapped buffer instead: the kernel reads its operands from host memory
    // and writes the result there, so a call is two host memcpy, one launch and one stream synchronisation -- no copy
    // engine work (three cudaMemcpyAsync cost more than the kernel at these sizes: 21 -> 14 us per call,
    // profiles/dropin_table_latency_r2.txt).
    char *h = nullptr, *h_dev = nullptr;
    size_t hcap = 0;
    int device = -1;
    PlanKey last_key;
    int32_t last_sent[4] = {0, 0, 0, 0};
    scgpu_ntt_plan *last_plan = nullptr;
    void *ensure(int i, size_t bytes)
    {
        if (!st && cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) dropin_fatal("stream");
        if (!d_rc && cudaMalloc(&d_rc, sizeof(int32_t)) != cudaSuccess) dropin_fatal("cudaMalloc");
        if (cap[i] < bytes) {
            if (d[i]) { cudaStreamSynchronize(st); cudaFree(d[i]); }
            size_t want = bytes < 8192 ? 8192 : bytes;
            if (cudaMalloc(&d[i], want) != cudaSuccess) dropin_fatal("cudaMalloc");
            cap[i] = want;
        }
        return d[i];
    }
    char *mapped(size_t bytes)
    {
        if (!st && cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) dropin_fatal("stream");
        if (hcap < bytes) {
            if (h) { cudaStreamSynchronize(st); cudaFreeHost(h); h = nullptr; }
            size_t want = bytes < 32768 ? 32768 : bytes;
            if (cudaHostAlloc(reinterpret_cast<void **>(&h), want, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess)
                dropin_fatal("cudaHostAlloc");
            if (cudaHostGetDevicePointer(reinterpret_cast<void **>(&h_dev), h, 0) != cudaSuccess) dropin_fatal("cudaHostGetDevicePointer");
            hcap = want;
        }
        return h;
    }
    ~ThreadCtx()
    {
        // errors are ignored: at process exit the context may already have been torn down
        if (device >= 0 && cudaSetDevice(device) == cudaSuccess) {
            if (st) cudaStreamSynchronize(st);
            if (h) cudaFreeHost(h);
            for (int i = 0; i < 3; i++) cudaFree(d[i]);
            cudaFree(d_rc);
            if (st) cudaStreamDestroy(st);
        }
        cudaGetLastError();
    }
    scgpu_ntt_plan *plan_for(const PlanKey &key)
    {
        if (last_plan && key == last_key) {
            int32_t sent[4];
            read_sentinels(key, sent);
            if (memcmp(sent, last_sent, sizeof(sent)) == 0) return last_plan;
        }
        last_plan = g_cache.get(key);
        last_key = key;
        read_sentinels(key, last_sent);
        return last_plan;
    }
};
thread_local ThreadCtx t_ctx;

// rows up to this size are read and written by the kernel in place in mapped host memory (ThreadCtx::mapped)
constexpr size_t kZeroCopyMax = 64 * 1024;
bool zero_copy_enabled()
{
    static const int on = [] { const char *e = getenv("SCGPU_DROPIN_ZERO_COPY"); return (e && atoi(e) == 0) ? 0 : 1; }();
    return on != 0;
}

// One reference call = one row through the batch kernel.
SINT32 run_one(int variant, int op, const ntt_params_t *p, size_t n, SINT32 *out, const void *a, const void *b,
               size_t b_elems, const void *w, const void *r, int tw_bits, int32_t scalar)
{
    ThreadCtx &c = t_ctx;
    PlanKey key;
    key.w = w; key.r = r; key.n = (uint64_t)n; key.inv = p->inv_q_dbl;
    key.q = p->u.ntt32.q; key.m = p->u.ntt32.m; key.k = p->u.ntt32.k;
    key.variant = variant; key.tw_bits = w ? tw_bits : 0; key.device = dropin_device();
    scgpu_ntt_plan *plan = c.plan_for(key);
    if (cudaSetDevice(plan->dev.device) != cudaSuccess) dropin_fatal("cudaSetDevice");
    c.device = plan->dev.device;
    const size_t abytes = n * a_elem_size(op), obytes = n * 4, bbytes = b_elems * b_elem_size(op);
    if (abytes + bbytes + obytes <= kZeroCopyMax && zero_copy_enabled()) {
        auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
        const size_t bo = up(abytes), oo = bo + up(b ? bbytes : 0), ro = oo + up(obytes);
        char *h = c.mapped(ro + 256);
        char *hd = c.h_dev;
        memcpy(h, a, abytes);
        if (b) memcpy(h + bo, b, bbytes);
        *reinterpret_cast<int32_t *>(h + ro) = 0;
        if (scgpu_ntt_batch(plan, op, reinterpret_cast<int32_t *>(hd + oo), hd, b ? hd + bo : nullptr, b_elems, 1, scalar,
                            reinterpret_cast<int32_t *>(hd + ro), c.st) != SCGPU_OK)
            dropin_fatal("kernel launch");
        if (cudaStreamSynchronize(c.st) != cudaSuccess) dropin_fatal("kernel");
        memcpy(out, h + oo, obytes);
        return (op == SCGPU_OP_INVERT || op == SCGPU_OP_DIV) ? *reinterpret_cast<int32_t *>(h + ro) : 0;
    }
    void *da = c.ensure(0, abytes);
    void *dout = c.ensure(1, obytes);
    void *db = b ? c.ensure(2, bbytes) : nullptr;
    bool ok = cudaMemcpyAsync(da, a, abytes, cudaMemcpyHostToDevice, c.st) == cudaSuccess;
    if (b) ok = ok && cudaMemcpyAsync(db, b, bbytes, cudaMemcpyHostToDevice, c.st) == cudaSuccess;
    if (!ok) dropin_fatal("H2D copy");
    if (scgpu_ntt_batch(plan, op, static_cast<int32_t *>(dout), da, db, b_elems, 1, scalar, c.d_rc, c.st) != SCGPU_OK)
        dropin_fatal("kernel launch");
    int32_t rc = 0;
    ok = cudaMemcpyAsync(out, dout, obytes, cudaMemcpyDeviceToHost, c.st) == cudaSuccess;
    if (op == SCGPU_OP_INVERT || op == SCGPU_OP_DIV)
        ok = ok && cudaMemcpyAsync(&rc, c.d_rc, sizeof(rc), cudaMemcpyDeviceToHost, c.st) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(c.st) == cudaSuccess;
    if (!ok) dropin_fatal("D2H copy");
    return rc;
}

[[noreturn]] void not_on_hot_path(const char *member)
{
    fprintf(stderr, "libscgpu: utils_arith_ntt_t::%s is not GPU backed: no scheme of the reference calls the SINT16-data "
                    "or limb-data members (SURVEY.md 3.6); use the *_32 members\n", member);
    abort();
}

template <int V>
struct DropIn {
    // scalars: one-element rows
    static SINT32 modn_32(SINT32 x, scP p) { SINT32 o; run_one(V, SCGPU_OP_MODN, p, 1, &o, &x, nullptr, 0, nullptr, nullptr, 0, 0); return o; }
    static SINT32 muln_32(SINT32 x, SINT32 y, scP p) { SINT32 o; run_one(V, SCGPU_OP_MULN, p, 1, &o, &x, &y, 1, nullptr, nullptr, 0, 0); return o; }
    static SINT32 sqrn_32(SINT32 x, scP p) { SINT32 o; run_one(V, SCGPU_OP_SQRN, p, 1, &o, &x, nullptr, 0, nullptr, nullptr, 0, 0); return o; }
    static SINT32 pwr_32(SINT32 x, SINT32 e, scP p) { SINT32 o; run_one(V, SCGPU_OP_PWR, p, 1, &o, &x, &e, 1, nullptr, nullptr, 0, 0); return o; }
    static void mul_32_sparse(SINT32 *v, size_t n, UINT16 omega, const SINT32 *t, const SINT32 *u)
    {
        ntt_params_t p; init_reduce(&p, n, 12289);      // the generic sparse product does not reduce (ntt.c:381-400)
        run_one(V, SCGPU_OP_SPARSE32, &p, n, v, t, u, omega, nullptr, nullptr, 0, omega);
    }
    static void mul_32_sparse_16(SINT32 *v, size_t n, UINT16 omega, const SINT16 *t, const SINT32 *u)
    {
        ntt_params_t p; init_reduce(&p, n, 12289);
        run_one(V, SCGPU_OP_SPARSE16, &p, n, v, t, u, omega, nullptr, nullptr, 0, omega);
    }
    static void mul_32_pointwise(SINT32 *v, scP p, const SINT32 *t, const SINT32 *u) { run_one(V, SCGPU_OP_PW, p, p->n, v, t, u, p->n, nullptr, nullptr, 0, 0); }
    static void mul_32_pointwise_16(SINT32 *v, scP p, const SINT32 *t, const SINT16 *u) { run_one(V, SCGPU_OP_PW16, p, p->n, v, t, u, p->n, nullptr, nullptr, 0, 0); }
    static void mul_32_scalar(SINT32 *v, scP p, const SINT32 *t, SINT32 c) { run_one(V, SCGPU_OP_SCALAR, p, p->n, v, t, nullptr, 0, nullptr, nullptr, 0, c); }
    static void fft_32_32(SINT32 *v, scP p, const SINT32 *w) { run_one(V, SCGPU_OP_FFT, p, p->n, v, v, nullptr, 0, w, nullptr, 32, 0); }
    static void fft_32_32_large(SINT32 *v, scP p, const SINT32 *w) { run_one(V, SCGPU_OP_FFT_LARGE, p, p->n, v, v, nullptr, 0, w, nullptr, 32, 0); }
    static void fft_32_16(SINT32 *v, scP p, const SINT16 *w) { run_one(V, SCGPU_OP_FFT, p, p->n, v, v, nullptr, 0, w, nullptr, 16, 0); }
    static void fft_32_16_large(SINT32 *v, scP p, const SINT16 *w) { run_one(V, SCGPU_OP_FFT_LARGE, p, p->n, v, v, nullptr, 0, w, nullptr, 16, 0); }
    static SINT32 invert_32(SINT32 *v, scP p, size_t n) { return run_one(V, SCGPU_OP_INVERT, p, n, v, v, nullptr, 0, nullptr, nullptr, 0, 0); }
    static SINT32 div_32(SINT32 *num, const SINT32 *den, scP p, size_t n) { return run_one(V, SCGPU_OP_DIV, p, n, num, num, den, n, nullptr, nullptr, 0, 0); }
    static void flip_32(SINT32 *v, scP p) { run_one(V, SCGPU_OP_FLIP, p, p->n, v, v, nullptr, 0, nullptr, nullptr, 0, 0); }
    static void center_32(SINT32 *v, size_t n, scP p) { run_one(V, SCGPU_OP_CENTER, p, n, v, v, nullptr, 0, nullptr, nullptr, 0, 0); }
    static void normalize_32(SINT32 *v, size_t n, scP p) { run_one(V, SCGPU_OP_NORMALIZE, p, n, v, v, nullptr, 0, nullptr, nullptr, 0, 0); }
    static void fwd_ntt_32_32(SINT32 *v, scP p, const SINT32 *t, const SINT32 *w) { run_one(V, SCGPU_OP_FWD, p, p->n, v, t, nullptr, 0, w, nullptr, 32, 0); }
    static void inv_ntt_32_32(SINT32 *v, scP p, const SINT32 *t, const SINT32 *w, const SINT32 *r) { run_one(V, SCGPU_OP_INV, p, p->n, v, t, nullptr, 0, w, r, 32, 0); }
    static void fwd_ntt_32_32_large(SINT32 *v, scP p, const SINT32 *t, const SINT32 *w) { run_one(V, SCGPU_OP_FWD_LARGE, p, p->n, v, t, nullptr, 0, w, nullptr, 32, 0); }
    static void inv_ntt_32_32_large(SINT32 *v, scP p, const SINT32 *t, const SINT32 *w, const SINT32 *r) { run_one(V, SCGPU_OP_INV_LARGE, p, p->n, v, t, nullptr, 0, w, r, 32, 0); }
    static void fwd_ntt_32_16(SINT32 *v, scP p, const SINT32 *t, const SINT16 *w) { run_one(V, SCGPU_OP_FWD, p, p->n, v, t, nullptr, 0, w, nullptr, 16, 0); }
    static void inv_ntt_32_16(SINT32 *v, scP p, const SINT32 *t, const SINT16 *w, const SINT16 *r) { run_one(V, SCGPU_OP_INV, p, p->n, v, t, nullptr, 0, w, r, 16, 0); }
    static void fwd_ntt_32_16_large(SINT32 *v, scP p, const SINT32 *t, const SINT16 *w) { run_one(V, SCGPU_OP_FWD_LARGE, p, p->n, v, t, nullptr, 0, w, nullptr, 16, 0); }
    static void inv_ntt_32_16_large(SINT32 *v, scP p, const SINT32 *t, const SINT16 *w, const SINT16 *r) { run_one(V, SCGPU_OP_INV_LARGE, p, p->n, v, t, nullptr, 0, w, r, 16, 0); }
};

// stubs for the 51 members no scheme calls
#define STUB(ret, name, args) static ret stub_##name args { not_on_hot_path(#name); }
STUB(SINT16, modn_16, (SINT16, scP)) STUB(SINT16, muln_16, (SINT16, SINT16, scP)) STUB(SINT16, sqrn_16, (SINT16, scP))
STUB(void, mul_16_sparse, (SINT16 *, size_t, UINT16, const SINT16 *, const SINT16 *))
STUB(void, mul_16_pointwise, (SINT16 *, scP, const SINT16 *, const SINT16 *))
STUB(void, mul_16_scalar, (SINT16 *, scP, const SINT16 *, SINT16))
STUB(void, fft_16, (SINT16 *, scP, const SINT16 *))
STUB(SINT32, pwr_16, (SINT16, SINT16, scP)) STUB(SINT32, invert_16, (SINT16 *, scP, size_t))
STUB(SINT32, div_16, (SINT16 *, const SINT16 *, scP, size_t))
STUB(void, flip_16, (SINT16 *, scP)) STUB(void, center_16, (SINT16 *, size_t, scP))
STUB(void, fwd_ntt_16, (SINT16 *, scP, const SINT16 *, const SINT16 *))
STUB(void, inv_ntt_16, (SINT16 *, scP, const SINT16 *, const SINT16 *, const SINT16 *))
STUB(sc_slimb_t, modn_limb, (sc_slimb_t, scP)) STUB(sc_slimb_t, muln_limb, (sc_slimb_t, sc_slimb_t, scP))
STUB(void, mul_limb_sparse, (sc_slimb_t *, size_t, UINT16, const SINT32 *, const sc_slimb_t *))
STUB(void, mul_limb_sparse_16, (sc_slimb_t *, size_t, UINT16, const SINT16 *, const sc_slimb_t *))
STUB(void, mul_limb_pointwise, (sc_slimb_t *, scP, const sc_slimb_t *, const sc_slimb_t *))
STUB(void, mul_limb_pointwise_32, (sc_slimb_t *, scP, const sc_slimb_t *, const SINT32 *))
STUB(void, mul_limb_pointwise_16, (sc_slimb_t *, scP, const sc_slimb_t *, const SINT16 *))
STUB(void, mul_limb_scalar, (sc_slimb_t *, scP, const sc_slimb_t *, sc_slimb_t))
STUB(void, fft_limb, (sc_slimb_t *, scP, const sc_slimb_t *))
STUB(void, fft_limb_32, (sc_slimb_t *, scP, const SINT32 *))
STUB(void, fft_limb_16, (sc_slimb_t *, scP, const SINT16 *))
STUB(SINT32, invert_limb, (sc_slimb_t *, scP, size_t))
STUB(SINT32, div_limb, (sc_slimb_t *, const sc_slimb_t *, scP, size_t))
STUB(void, flip_limb, (sc_slimb_t *, scP)) STUB(void, center_limb, (sc_slimb_t *, size_t, scP))
STUB(void, fwd_ntt_limb, (sc_slimb_t *, scP, const sc_slimb_t *, const sc_slimb_t *))
STUB(void, inv_ntt_limb, (sc_slimb_t *, scP, const sc_slimb_t *, const sc_slimb_t *, const sc_slimb_t *))
STUB(void, fwd_ntt_limb_32, (sc_slimb_t *, scP, const sc_slimb_t *, const SINT32 *))
STUB(void, inv_ntt_limb_32, (sc_slimb_t *, scP, const sc_slimb_t *, const SINT32 *, const SINT32 *))
STUB(void, fwd_ntt_limb_16, (sc_slimb_t *, scP, const sc_slimb_t *, const SINT16 *))
STUB(void, inv_ntt_limb_16, (sc_slimb_t *, scP, const sc_slimb_t *, const SINT16 *, const SINT16 *))
#undef STUB

template <int V>
utils_arith_ntt_t make_table()
{
    utils_arith_ntt_t t;
    t.modn_16 = stub_modn_16; t.muln_16 = stub_muln_16; t.sqrn_16 = stub_sqrn_16;
    t.mul_16_sparse = stub_mul_16_sparse; t.mul_16_pointwise = stub_mul_16_pointwise; t.mul_16_scalar = stub_mul_16_scalar;
    t.fft_16 = stub_fft_16; t.large_fft_16 = stub_fft_16;
    t.pwr_16 = stub_pwr_16; t.invert_16 = stub_invert_16; t.div_16 = stub_div_16; t.flip_16 = stub_flip_16;
    t.center_16 = stub_center_16; t.normalize_16 = stub_center_16;
    t.fwd_ntt_16 = stub_fwd_ntt_16; t.inv_ntt_16 = stub_inv_ntt_16; t.fwd_ntt_16_large = stub_fwd_ntt_16; t.inv_ntt_16_large = stub_inv_ntt_16;

    using D = DropIn<V>;
    t.modn_32 = D::modn_32; t.muln_32 = D::muln_32; t.sqrn_32 = D::sqrn_32;
    t.mul_32_sparse = D::mul_32_sparse; t.mul_32_sparse_16 = D::mul_32_sparse_16;
    t.mul_32_pointwise = D::mul_32_pointwise; t.mul_32_pointwise_16 = D::mul_32_pointwise_16; t.mul_32_scalar = D::mul_32_scalar;
    t.fft_32_32 = D::fft_32_32; t.fft_32_32_large = D::fft_32_32_large; t.fft_32_16 = D::fft_32_16; t.fft_32_16_large = D::fft_32_16_large;
    t.pwr_32 = D::pwr_32; t.invert_32 = D::invert_32; t.div_32 = D::div_32; t.flip_32 = D::flip_32;
    t.center_32 = D::center_32; t.normalize_32 = D::normalize_32;
    t.fwd_ntt_32_32 = D::fwd_ntt_32_32; t.inv_ntt_32_32 = D::inv_ntt_32_32;
    t.fwd_ntt_32_32_large = D::fwd_ntt_32_32_large; t.inv_ntt_32_32_large = D::inv_ntt_32_32_large;
    t.fwd_ntt_32_16 = D::fwd_ntt_32_16; t.inv_ntt_32_16 = D::inv_ntt_32_16;
    t.fwd_ntt_32_16_large = D::fwd_ntt_32_16_large; t.inv_ntt_32_16_large = D::inv_ntt_32_16_large;

    t.modn_limb = stub_modn_limb; t.muln_limb = stub_muln_limb; t.sqrn_limb = stub_modn_limb;
    t.mul_limb_sparse = stub_mul_limb_sparse; t.mul_limb_sparse_16 = stub_mul_limb_sparse_16;
    t.mul_limb_pointwise = stub_mul_limb_pointwise; t.mul_limb_pointwise_32 = stub_mul_limb_pointwise_32;
    t.mul_limb_pointwise_16 = stub_mul_limb_pointwise_16; t.mul_limb_scalar = stub_mul_limb_scalar;
    t.fft_limb = stub_fft_limb; t.fft_limb_large = stub_fft_limb; t.fft_limb_32 = stub_fft_limb_32; t.fft_limb_32_large = stub_fft_limb_32;
    t.fft_limb_16 = stub_fft_limb_16; t.fft_limb_16_large = stub_fft_limb_16;
    t.pwr_limb = stub_muln_limb; t.invert_limb = stub_invert_limb; t.div_limb = stub_div_limb; t.flip_limb = stub_flip_limb;
    t.center_limb = stub_center_limb; t.normalize_limb = stub_center_limb;
    t.fwd_ntt_limb = stub_fwd_ntt_limb; t.inv_ntt_limb = stub_inv_ntt_limb;
    t.fwd_ntt_limb_large = stub_fwd_ntt_limb; t.inv_ntt_limb_large = stub_inv_ntt_limb;
    t.fwd_ntt_limb_32 = stub_fwd_ntt_limb_32; t.inv_ntt_limb_32 = stub_inv_ntt_limb_32;
    t.fwd_ntt_limb_32_large = stub_fwd_ntt_limb_32; t.inv_ntt_limb_32_large = stub_inv_ntt_limb_32;
    t.fwd_ntt_limb_16 = stub_fwd_ntt_limb_16; t.inv_ntt_limb_16 = stub_inv_ntt_limb_16;
    t.fwd_ntt_limb_16_large = stub_fwd_ntt_limb_16; t.inv_ntt_limb_16_large = stub_inv_ntt_limb_16;
    return t;
}

const utils_arith_ntt_t g_tab_reference = make_table<V_REFERENCE>();
const utils_arith_ntt_t g_tab_barrett = make_table<V_BARRETT>();
const utils_arith_ntt_t g_tab_fp = make_table<V_FP>();
const utils_arith_ntt_t g_tab_avx = make_table<V_AVX>();
const utils_arith_ntt_t g_tab_7681 = make_table<V_SOL7681>();
const utils_arith_ntt_t g_tab_8380417 = make_table<V_SOL8380417>();

}  // namespace

extern "C" {
const utils_arith_ntt_t *ntt_table = nullptr;      // ntt.c:31

// arith.c:360-396: unknown types select the reference table
const utils_arith_ntt_t *utils_arith_ntt(safecrypto_ntt_e type)
{
    switch (type) {
    case SC_NTT_BARRETT:         ntt_table = &g_tab_barrett; break;
    case SC_NTT_FLOATING_POINT:  ntt_table = &g_tab_fp; break;
    case SC_NTT_AVX:             ntt_table = &g_tab_avx; break;
    case SC_NTT_SOLINAS_7681:    ntt_table = &g_tab_7681; break;
    case SC_NTT_SOLINAS_8380417: ntt_table = &g_tab_8380417; break;
    default:                     ntt_table = &g_tab_reference; break;
    }
    return ntt_table;
}
}
