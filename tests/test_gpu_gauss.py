"""Parity of the CUDA sampler / CSPRNG path with the CPU oracle: bit-exact samples for the same seeds."""
import ctypes
import os

import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import libsafecrypto_b200 as sc  # noqa: E402

G = O.golden("golden_v1")
DEV = "cuda:0"


def seeds_for(count, length=64, salt=0):
    return np.array([[(s * 131 + j * 7 + 3 + salt) & 0xFF for j in range(length)] for s in range(count)], dtype=np.uint8)


def gpu_words(prng, seeds, nwords, seed_period=0):
    d_seeds = torch.from_numpy(seeds).to(DEV)
    out = torch.zeros((seeds.shape[0], nwords), dtype=torch.int32, device=DEV)
    st = sc.lib().scgpu_prng_words(prng, d_seeds.data_ptr(), seeds.shape[1], seed_period, seeds.shape[0], nwords,
                                   out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert st == 0, sc.lib().scgpu_last_error()
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.uint32)


def gpu_samples(sampler, precision, blinding, prng, tail, sigma, seeds, n, calls=1, centre=0, discard=0):
    plan = sc.GaussPlan(sampler, precision, blinding, tail, sigma)
    d_seeds = torch.from_numpy(seeds).to(DEV)
    out = torch.full((seeds.shape[0], n * calls), 123456, dtype=torch.int32, device=DEV)
    plan.streams(prng, d_seeds, n, out, calls=calls, centre=centre, discard=discard)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_prng_word_stream(prng):
    seeds = seeds_for(5)
    got = gpu_words(prng, seeds, 10000)
    for i in range(seeds.shape[0]):
        assert np.array_equal(got[i], O.port().prng_words(prng, seeds[i].tobytes(), 10000))
    name = "chacha" if prng == O.PRNG_CHACHA else "aes"
    gold = G["prng_%s_words" % name]
    assert np.array_equal(gpu_words(prng, G["prng_seed"].reshape(1, -1), gold.size)[0], gold)


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_prng_reseed_boundaries(prng):
    seeds = seeds_for(2, 48, salt=9)
    got = gpu_words(prng, seeds, 3 * 4096 + 5, seed_period=64)
    for i in range(2):
        assert np.array_equal(got[i], O.port().prng_words(prng, seeds[i].tobytes(), 3 * 4096 + 5, seed_period=64))


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("blinding", [O.NORMAL_SAMPLES, O.BLINDING_SAMPLES, O.SHUFFLE_SAMPLES])
def test_cdf_vectors(prng, precision, blinding):
    seeds = seeds_for(70)
    for discard, n, calls, centre in ((0, 512, 2, 3), (2, 512, 1, 0), (6, 256, 2, -1), (0, 77, 3, 0), (0, 1, 1, 5)):
        got = gpu_samples(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, n, calls, centre, discard)
        exp = O.port().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, n,
                                     discard=discard, centre=centre, calls=calls)
        assert np.array_equal(got, exp), (discard, n, calls)


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("precision", [128, 192])
def test_high_precision_cdf_vectors(prng, precision):
    """128 / 192-bit CDF sampling over a caller-built table (scgpu_gauss_plan_create_table): every vector mode,
    discard, several calls; plus the golden samples of the compiled reference; 256-bit is refused."""
    seeds = seeds_for(37)
    pname = "chacha" if prng == O.PRNG_CHACHA else "aes"
    G2 = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v2.npz"))

    def run(table, blinding, sd, n, calls=1, centre=0, discard=0):
        plan = sc.GaussPlan(sc.SAMPLER_CDF, precision, blinding, 0.0, 0.0, table=table)
        out = torch.full((sd.shape[0], n * calls), 123456, dtype=torch.int32, device=DEV)
        plan.streams(prng, torch.from_numpy(sd).to(DEV), n, out, calls=calls, centre=centre, discard=discard)
        torch.cuda.synchronize()
        return out.cpu().numpy()

    for blinding in (O.NORMAL_SAMPLES, O.BLINDING_SAMPLES, O.SHUFFLE_SAMPLES):
        tab = O.high_precision_cdf_table(precision, 13.42, 215.0, blinding)
        O.port().set_high_table(precision, tab)
        for discard, n, calls, centre in ((0, 512, 2, 3), (4, 200, 1, 0), (0, 1, 3, -7)):
            exp = O.port().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, n,
                                         discard=discard, centre=centre, calls=calls)
            assert np.array_equal(run(tab, blinding, seeds, n, calls, centre, discard), exp), (blinding, discard, n)
        g = G2["cdf%d_b%d_sigma4p5" % (precision, blinding)]
        got = run(g, blinding, G2["gauss_seeds"], 256, calls=2, discard=(2 if blinding == 2 else 0))
        assert np.array_equal(got, G2["gauss_cdf%d_%s_b%d" % (precision, pname, blinding)])
    got = run(G2["cdf%d_own_sigma4p5" % precision], 0, G2["gauss_seeds"], 64)
    assert np.array_equal(got, G2["gauss_cdf%d_%s_own" % (precision, pname)])
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_CDF, 256, 0, 0.0, 0.0, table=np.zeros((64, 4), dtype=np.uint64))


@pytest.mark.parametrize("pname,prng", [("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)])
def test_golden_samples_on_gpu(pname, prng):
    seeds = G["gauss_seeds"]
    for bl in (0, 1, 2):
        for prec in (32, 64):
            got = gpu_samples(O.SAMPLER_CDF, prec, bl, prng, 13.42, 215.0, seeds, 512, calls=2)
            assert np.array_equal(got, G["gauss_cdf%d_%s_b%d" % (prec, pname, bl)])
    got = gpu_samples(O.SAMPLER_CDF, 64, 0, prng, 13.42, 215.0, seeds, 512, discard=4)
    assert np.array_equal(got, G["gauss_cdf64_%s_discard" % pname])
    for key, smp, tail, sigma, n in (("ky64", O.SAMPLER_KNUTH_YAO, 13.42, 215.0, 128), ("ky64s", O.SAMPLER_KNUTH_YAO, 13.0, 4.5, 512),
                                     ("ber64", O.SAMPLER_BERNOULLI, 13.42, 215.0, 128), ("ber64s", O.SAMPLER_BERNOULLI, 13.0, 4.5, 512)):
        got = gpu_samples(smp, 64, 0, prng, tail, sigma, seeds, n)
        assert np.array_equal(got, G["gauss_%s_%s" % (key, pname)]), key


def test_survey_anchor_samples_on_gpu():
    ent = np.array([[(i * 7 + 3) & 0xFF for i in range(64)]], dtype=np.uint8)
    c = gpu_samples(O.SAMPLER_CDF, 64, 0, O.PRNG_CHACHA, 13.42, 215.0, ent, 12)[0]
    a = gpu_samples(O.SAMPLER_CDF, 64, 0, O.PRNG_AES_CTR_DRBG, 13.42, 215.0, ent, 12)[0]
    assert list(c) == [0, 0, -251, 248, 113, 96, -138, 17, -341, 64, -399, -212]
    assert list(a) == [-319, 333, 125, -307, -208, 85, -140, -269, -1, 74, -120, 180]


@pytest.mark.parametrize("sampler,precision", [(O.SAMPLER_KNUTH_YAO, 64), (O.SAMPLER_KNUTH_YAO, 32), (O.SAMPLER_KNUTH_YAO, 128),
                                               (O.SAMPLER_BERNOULLI, 64)])
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("tail,sigma,n", [(13.42, 215.0, 96), (13.0, 4.5, 512)])
def test_ky_bernoulli_samples(sampler, precision, prng, tail, sigma, n):
    seeds = seeds_for(40, salt=1)
    got = gpu_samples(sampler, precision, 0, prng, tail, sigma, seeds, n)
    exp = O.port().gauss_streams(sampler, precision, 0, prng, tail, sigma, seeds, n)
    assert np.array_equal(got, exp)
    if O.ref_available():
        assert np.array_equal(exp, O.ref().gauss_streams(sampler, precision, 0, prng, tail, sigma, seeds, n))


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_ky_bernoulli_vector_modes_and_ragged_batches(prng):
    """Knuth-Yao (rank / select walk) and Bernoulli (one-draw-per-trip lanes) beyond the plain case: stream counts
    that are not a multiple of a warp or a CTA, several calls, a centre, discard, and the shuffle / blinding vector
    wrappers (sampler-agnostic in the reference, sampling.c:127-191; Knuth-Yao's blinding table is built from
    sigma / sqrt 2, gaussian_knuth_yao.c:144-146, checked against the compiled reference's table)."""
    for count in (1, 33, 130):
        seeds = seeds_for(count, 44, salt=count)
        for sampler, prec in ((O.SAMPLER_KNUTH_YAO, 64), (O.SAMPLER_BERNOULLI, 64)):
            for discard, n, calls, centre in ((0, 50, 2, 3), (4, 37, 1, 0), (6, 5, 3, -7)):
                got = gpu_samples(sampler, prec, 0, prng, 13.42, 215.0, seeds, n, calls=calls, centre=centre, discard=discard)
                exp = O.port().gauss_streams(sampler, prec, 0, prng, 13.42, 215.0, seeds, n, discard=discard, centre=centre, calls=calls)
                assert np.array_equal(got, exp), (count, sampler, discard)
    seeds = seeds_for(9, 40, salt=5)
    for sampler, prec, tail, sigma in ((O.SAMPLER_KNUTH_YAO, 64, 13.0, 19.53), (O.SAMPLER_KNUTH_YAO, 32, 13.0, 4.5), (O.SAMPLER_BERNOULLI, 64, 13.0, 19.53)):
        for blinding in (O.SHUFFLE_SAMPLES, O.BLINDING_SAMPLES):
            for discard, n in ((0, 64), (2, 77)):
                got = gpu_samples(sampler, prec, blinding, prng, tail, sigma, seeds, n, calls=2, centre=1, discard=discard)
                exp = O.port().gauss_streams(sampler, prec, blinding, prng, tail, sigma, seeds, n, discard=discard, centre=1, calls=2)
                assert np.array_equal(got, exp), (sampler, blinding, discard)
    if O.ref_available():
        for bw in (32, 64, 128):
            a, ba = O.port().ky_table(bw, 13.42, 215.0, 1)
            b, bb = O.ref().ky_table(bw, 13.42, 215.0, 1)
            assert ba == bb and np.array_equal(a, b)


@pytest.mark.skipif(not O.ref_available(), reason="the look-up tables are constants of the reference: read from oracle/_ref/libscref.so")
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("dimension", [256, 512])
def test_knuth_yao_fast_over_the_references_tables(prng, dimension):
    """gaussian_knuth_yao_fast_sample (gaussian_knuth_yao_fast.c:303-368): the tables are read out of the compiled
    reference at run time and handed to scgpu_gauss_plan_create_ky_fast; samples against the reference's own."""
    tabs = O.ref().kyfast_tables(dimension)
    plan = sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, 0, 0.0, 0.0, ky_fast=tabs)
    seeds = seeds_for(70, 40, salt=dimension)
    for n, calls, centre in ((512, 2, 0), (77, 1, 5)):
        out = torch.full((seeds.shape[0], n * calls), 99, dtype=torch.int32, device=DEV)
        plan.streams(prng, torch.from_numpy(seeds).to(DEV), n, out, calls=calls, centre=centre)
        torch.cuda.synchronize()
        exp = O.ref().gauss_streams(O.SAMPLER_KNUTH_YAO_FAST, dimension, 0, prng, 0.0, 0.0, seeds, n, centre=centre, calls=calls)
        assert np.array_equal(out.cpu().numpy(), exp)
        if n == 512:        # sanity: sigma 4.512 / 4.8591 (a ChaCha20 stream opens with three zero words, skip them)
            assert abs(out.cpu().numpy()[:, 16:].std() - (4.51 if dimension == 256 else 4.86)) < 0.2
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, 1, 0.0, 0.0, ky_fast=tabs)         # blinding: refused as configure_sampler does


def test_bernoulli_and_knuth_yao_at_scale():
    """2^13 streams x 256 samples of each: every sample against the port, moments as a sanity check."""
    seeds = np.random.default_rng(11).integers(0, 256, size=(1 << 13, 40)).astype(np.uint8)
    for sampler, lo, hi in ((O.SAMPLER_BERNOULLI, 205.0, 225.0), (O.SAMPLER_KNUTH_YAO, 150.0, 260.0)):
        got = gpu_samples(sampler, 64, 0, O.PRNG_CHACHA, 13.42, 215.0, seeds, 256)
        exp = O.port().gauss_streams(sampler, 64, 0, O.PRNG_CHACHA, 13.42, 215.0, seeds, 256)
        assert np.array_equal(got, exp)
        assert abs(got.mean()) < 2.0 and lo < got.std() < hi, (sampler, got.std())


def test_sampling_statistics_at_scale():
    """2^14 streams x 512 samples: moments of the CDF sampler, and determinism of a re-run."""
    rng = np.random.default_rng(5)
    seeds = rng.integers(0, 256, size=(1 << 14, 40)).astype(np.uint8)
    for prng in (O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG):
        x = gpu_samples(O.SAMPLER_CDF, 64, 0, prng, 13.42, 215.0, seeds, 512)
        assert abs(x.mean()) < 0.5 and abs(x.std() - 215.0) < 0.5 and np.abs(x).max() < 4096
        assert np.array_equal(x, gpu_samples(O.SAMPLER_CDF, 64, 0, prng, 13.42, 215.0, seeds, 512))
        sl = slice(5000, 5016)
        assert np.array_equal(x[sl], O.port().gauss_streams(O.SAMPLER_CDF, 64, 0, prng, 13.42, 215.0, seeds[sl], 512))


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("precision,tail,sigma", [(64, 13.42, 215.0), (32, 13.42, 215.0), (64, 13.0, 4.5), (32, 9.0, 1000.0),
                                                  (64, 9.0, 1000.0)])     # 128 KiB table: beside the AES tables it no longer fits
def test_throughput_kernels_against_the_port_in_bulk(prng, precision, tail, sigma):
    """The throughput kernels, first with the default fixed probe sequence, then with the optional guide table
    (cdf_search_guided): several million samples per (generator, precision, table) against the port's fixed-step
    search, every sample compared.  sigma = 4.5: a 64-entry table (most guide buckets empty or shared);
    sigma = 1000: the bracket is wide."""
    rng = np.random.default_rng(int(sigma * 10) + precision)
    big = sigma > 500 and precision == 64
    seeds = rng.integers(0, 256, size=(300 if big else 3000, 40)).astype(np.uint8)
    n = 1024
    got = gpu_samples(O.SAMPLER_CDF, precision, 0, prng, tail, sigma, seeds, n)
    exp = O.port().gauss_streams(O.SAMPLER_CDF, precision, 0, prng, tail, sigma, seeds, n)
    assert np.array_equal(got, exp)
    assert np.abs(got).max() > 3.5 * sigma            # the tails were visited
    old = sc.lib().scgpu_set_fixed_probe_search(0)    # guide-bracketed bisection: same samples
    assert old == 1                                   # constant-time lookups are the default
    try:
        assert np.array_equal(gpu_samples(O.SAMPLER_CDF, precision, 0, prng, tail, sigma, seeds, n), exp)
    finally:
        sc.lib().scgpu_set_fixed_probe_search(old)


def test_dropin_sampler_api():
    """create_sampler / get_vector_32 / prng_* with the reference's signatures, interleaving host draws
    (prng_32, prng_var) with device-side sampling on the same context."""
    L = sc.lib()
    L.prng_create.restype = ctypes.c_void_p
    L.prng_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t]
    L.prng_set_entropy.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
    L.prng_init.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
    L.prng_32.restype = ctypes.c_uint32
    L.prng_32.argtypes = [ctypes.c_void_p]
    L.prng_var.restype = ctypes.c_uint32
    L.prng_var.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
    L.prng_destroy.argtypes = [ctypes.c_void_p]
    L.create_sampler.restype = ctypes.c_void_p
    L.create_sampler.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int32, ctypes.c_int, ctypes.c_void_p,
                                 ctypes.c_float, ctypes.c_float]
    L.get_vector_32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_float]
    L.get_sample.argtypes = [ctypes.c_void_p]
    L.get_sample.restype = ctypes.c_int32
    L.destroy_sampler.argtypes = [ctypes.POINTER(ctypes.c_void_p)]
    seed = bytes(((i * 7 + 3) & 0xFF) for i in range(64))
    for prng in (O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG):
        ctx = L.prng_create(5, prng, 0, 0x00100000)          # SC_ENTROPY_USER_PROVIDED
        assert ctx
        assert L.prng_set_entropy(ctx, seed, len(seed)) == 0 and L.prng_init(ctx, b"SAFEcrypto nonce", 16) == 0
        smp = L.create_sampler(0, 64, 0, 512, 0, ctx, 13.42, 215.0)
        assert smp
        v1 = np.zeros(512, dtype=np.int32)
        L.get_vector_32(smp, v1.ctypes.data, 512, 0.0)
        words = [L.prng_32(ctx) for _ in range(3)]
        bits = L.prng_var(ctx, 5)
        single = L.get_sample(smp)
        v2 = np.zeros(100, dtype=np.int32)
        L.get_vector_32(smp, v2.ctypes.data, 100, 2.0)
        # the same call sequence on the oracle: 512 samples = 1024 words, then 3 words, 5 bits (1 word), ...
        script = [(64, 0)] * 512 + [(32, 0)] * 3 + [(0, 5)] + [(64, 0)] * 101
        raw = O.port().prng_script(prng, seed, script)
        tab = O.port().cdf_table(64, 0, 13.42, 215.0)

        def cdf(hi, lo):
            x = (int(hi) << 32) | int(lo)
            a = 0
            st = tab.size >> 1
            while st:
                if a + st < tab.size and int(tab[a + st]) < x:
                    a += st
                st >>= 1
            return a if x & 1 else -a
        exp1 = [cdf(raw[2 * i], raw[2 * i + 1]) for i in range(512)]
        assert list(v1) == exp1
        assert words == [int(x) for x in raw[1024:1027]] and bits == int(raw[1027])
        rest = raw[1028:]
        assert single == cdf(rest[0], rest[1])
        assert list(v2) == [cdf(rest[2 + 2 * i], rest[3 + 2 * i]) + 2 for i in range(100)]
        h = ctypes.c_void_p(smp)
        assert L.destroy_sampler(ctypes.byref(h)) == 0
        L.prng_destroy(ctx)
        # 128 / 192-bit CDF through the drop-in (func_alg_bliss_b.c:118 asks for SAMPLING_128BIT): the table is built by the
        # library (csrc/cdf_hp.cu), the samples are those of the port's sampler over that table on the same word stream
        for precision in (128, 192):
            ctx = L.prng_create(5, prng, 0, 0x00100000)
            assert L.prng_set_entropy(ctx, seed, len(seed)) == 0 and L.prng_init(ctx, b"SAFEcrypto nonce", 16) == 0
            smp = L.create_sampler(0, precision, 0, 512, 0, ctx, 13.42, 215.0)
            assert smp, precision
            v = np.zeros(300, dtype=np.int32)
            L.get_vector_32(smp, v.ctypes.data, 300, 0.0)
            nent = ctypes.c_size_t(0)
            assert L.scgpu_gauss_cdf_table_high(None, 0, ctypes.byref(nent), precision, 0, 13.42, 215.0) == 0
            tabh = np.zeros((nent.value, precision // 64), dtype=np.uint64)
            assert L.scgpu_gauss_cdf_table_high(tabh.ctypes.data, nent.value, ctypes.byref(nent), precision, 0, 13.42, 215.0) == 0
            O.port().set_high_table(precision, tabh)
            sd = np.frombuffer(seed, dtype=np.uint8)[None, :].copy()
            exp = O.port().gauss_streams(O.SAMPLER_CDF, precision, 0, prng, 13.42, 215.0, sd, 300)
            assert np.array_equal(v, exp[0]), precision
            h = ctypes.c_void_p(smp)
            assert L.destroy_sampler(ctypes.byref(h)) == 0
            L.prng_destroy(ctx)
        ctx = L.prng_create(5, prng, 0, 0x00100000)
        assert L.prng_set_entropy(ctx, seed, len(seed)) == 0 and L.prng_init(ctx, b"SAFEcrypto nonce", 16) == 0
        assert not L.create_sampler(0, 256, 0, 512, 0, ctx, 13.42, 215.0)      # the reference's 256-bit sampler reads an uninitialised word
        L.prng_destroy(ctx)


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/libscref.so not built")
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_mw_bootstrap_against_the_reference(prng):
    """Micciancio-Walter bootstrap (mw_bootstrap.c through create_sampler(.., SAMPLING_MW_BOOTSTRAP, ..)): arbitrary sigma
    and real-valued centres from the sigma-16 CDF base sampler; get_vector_32's clamped vectors and the per-sample
    centres of get_bootstrap_sample, against the compiled reference making the same calls."""
    plan = sc.GaussPlan(sc.SAMPLER_CDF, 64, 0, 13.0, 0.0, mw=True)
    seeds = seeds_for(48, 40, salt=3)
    d_seeds = torch.from_numpy(seeds).to(DEV)
    for sigma, centre, n in ((100.0, 0.3, 300), (215.0, -7.625, 128), (19.0, 1000.5, 64), (40.0, 0.0, 33)):
        out = torch.zeros((seeds.shape[0], n), dtype=torch.int32, device=DEV)
        plan.mw_streams(prng, d_seeds, n, out, sigma, centre)
        torch.cuda.synchronize()
        exp = O.ref().mw_streams(prng, seeds, n, 13.0, sigma, centre)
        assert np.array_equal(out.cpu().numpy(), exp), (sigma, centre)
    got = out.cpu().numpy()
    assert abs(got.std() - 40.0) < 3.0 and abs(got.mean()) < 3.0
    rng = np.random.default_rng(4)
    n = 200
    centres = rng.uniform(-50, 50, size=(seeds.shape[0], n)).astype(np.float32)
    out = torch.zeros((seeds.shape[0], n), dtype=torch.int32, device=DEV)
    plan.mw_streams(prng, d_seeds, n, out, 60.0, 0.0, centres=torch.from_numpy(centres).to(DEV))
    torch.cuda.synchronize()
    exp = O.ref().mw_streams(prng, seeds, n, 13.0, 60.0, sigmas=np.full(centres.shape, 60.0, np.float32), centres=centres)
    assert np.array_equal(out.cpu().numpy(), exp)            # the tail (13 sigma) never clamps here
    with pytest.raises(sc.ScgpuError):                        # below the network's own noise floor
        plan.mw_streams(prng, d_seeds, 4, out, 10.0, 0.0)


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/libscref.so not built")
def test_mw_bootstrap_dropin_api():
    """create_sampler(CDF, 64-bit, NORMAL, n, SAMPLING_MW_BOOTSTRAP, ..): get_vector_32, get_bootstrap_sample with varying
    sigma and centre, get_sample (the base sampler) and prng_32 interleaved on one context -- the same calls on libscref."""
    results = []
    seed = bytes(((i * 11 + 5) & 0xFF) for i in range(48))
    for L in (sc.lib(), O.ref().lib):
        L.prng_create.restype = ctypes.c_void_p
        L.prng_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t]
        L.prng_set_entropy.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
        L.prng_init.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
        L.prng_32.restype = ctypes.c_uint32
        L.prng_32.argtypes = [ctypes.c_void_p]
        L.prng_destroy.argtypes = [ctypes.c_void_p]
        L.create_sampler.restype = ctypes.c_void_p
        L.create_sampler.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int32, ctypes.c_int, ctypes.c_void_p,
                                     ctypes.c_float, ctypes.c_float]
        L.get_vector_32.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_float]
        L.get_bootstrap_sample.argtypes = [ctypes.c_void_p, ctypes.c_float, ctypes.c_float]
        L.get_bootstrap_sample.restype = ctypes.c_int32
        L.get_sample.argtypes = [ctypes.c_void_p]
        L.get_sample.restype = ctypes.c_int32
        L.destroy_sampler.argtypes = [ctypes.POINTER(ctypes.c_void_p)]
        ctx = L.prng_create(5, O.PRNG_AES_CTR_DRBG, 0, 0x00100000)
        assert ctx and L.prng_set_entropy(ctx, seed, len(seed)) == 0 and L.prng_init(ctx, b"SAFEcrypto nonce", 16) == 0
        smp = L.create_sampler(0, 64, 0, 256, 1, ctx, 13.0, 150.0)          # SAMPLING_MW_BOOTSTRAP = 1
        assert smp
        got = []
        v = np.zeros(256, dtype=np.int32)
        L.get_vector_32(smp, v.ctypes.data, 256, 2.75)
        got += list(v)
        got.append(L.prng_32(ctx))
        for sg, ce in ((33.5, 0.25), (90.0, -3.5), (500.0, 17.125), (20.0, 1e4)):
            got.append(L.get_bootstrap_sample(smp, sg, ce))
        got.append(L.get_sample(smp))
        L.get_vector_32(smp, v.ctypes.data, 100, -0.5)
        got += list(v[:100])
        h = ctypes.c_void_p(smp)
        assert L.destroy_sampler(ctypes.byref(h)) == 0
        L.prng_destroy(ctx)
        results.append([int(x) for x in got])
    assert results[0] == results[1]


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("precision,tail,sigma", [(128, 13.42, 215.0), (192, 10.0, 19.53), (128, 12.0, 4.5)])
def test_high_precision_cdf_table_built_by_the_library(prng, precision, tail, sigma):
    """scgpu_gauss_plan_create(CDF, 128 | 192, ...) builds the table of gauss_cdf_create_high_precision itself
    (csrc/cdf_hp.cu; pinned in tests/test_cdf_high.py): the samples are those of the port's sampler over that table,
    in every vector mode (blinding scales sigma inside the table construction, gaussian_cdf.c:225-228)."""
    import ctypes
    seeds = seeds_for(29, 40, salt=precision)
    for blinding in (O.NORMAL_SAMPLES, O.BLINDING_SAMPLES, O.SHUFFLE_SAMPLES):
        nent = ctypes.c_size_t(0)
        assert sc.lib().scgpu_gauss_cdf_table_high(None, 0, ctypes.byref(nent), precision, blinding, tail, sigma) == 0
        tab = np.zeros((nent.value, precision // 64), dtype=np.uint64)
        assert sc.lib().scgpu_gauss_cdf_table_high(tab.ctypes.data, nent.value, ctypes.byref(nent), precision, blinding, tail, sigma) == 0
        O.port().set_high_table(precision, tab)
        plan = sc.GaussPlan(sc.SAMPLER_CDF, precision, blinding, tail, sigma)
        for n, calls, centre, discard in ((256, 2, 0, 0), (33, 1, -4, 4)):
            out = torch.full((seeds.shape[0], n * calls), 777, dtype=torch.int32, device=DEV)
            plan.streams(prng, torch.from_numpy(seeds).to(DEV), n, out, calls=calls, centre=centre, discard=discard)
            torch.cuda.synchronize()
            exp = O.port().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, tail, sigma, seeds, n,
                                         discard=discard, centre=centre, calls=calls)
            assert np.array_equal(out.cpu().numpy(), exp), (blinding, n)
        if blinding == O.NORMAL_SAMPLES and sigma > 100:
            x = out.cpu().numpy()
            plan2 = sc.GaussPlan(sc.SAMPLER_CDF, precision, 0, tail, sigma)
            big = torch.empty((seeds.shape[0], 2048), dtype=torch.int32, device=DEV)
            plan2.streams(prng, torch.from_numpy(seeds).to(DEV), 2048, big)
            torch.cuda.synchronize()
            y = big.cpu().numpy()[:, 16:]
            assert abs(y.std() - sigma) < 0.02 * sigma and abs(y.mean()) < 0.05 * sigma
