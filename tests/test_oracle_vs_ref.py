"""Pin the C restatement (oracle/sc_oracle*.c) to the compiled reference (oracle/_ref/libscref.so).

Runs wherever oracle/_ref/libscref.so exists (built by oracle/Makefile from the reference's sources).
Without it the tests that need the library skip -- the committed fixtures in tests/golden/ then carry
the pin (tests/test_oracle_golden.py) -- and the table and anchor tests check the port against the
reference's outputs stored in the repository.
"""
import hashlib

import numpy as np
import pytest

import _oracle as O

needs_ref = pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref/libscref.so not built")

PARAMS = [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32), (8399873, 512, 32)]


def variants_for(q):
    v = [O.REFERENCE, O.BARRETT, O.FP, O.AVX]
    if q == 7681:
        v.append(O.SOLINAS_7681)
    if q == 8380417:
        v.append(O.SOLINAS_8380417)
    return v


def rand_inputs(rng, kind, q, shape):
    if kind == "uniform":
        return rng.integers(0, q, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "small":
        return rng.integers(-300, 301, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "lazy":          # the range a forward transform leaves behind
        return rng.integers(-70000, q * 600, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "signed":
        return rng.integers(-q + 1, q, size=shape, dtype=np.int64).astype(np.int32)
    raise ValueError(kind)


@pytest.mark.parametrize("tw_bits,q,n", O.TABLE_PARAMS)
def test_tables_match_generated(tw_bits, q, n):
    """The port's twiddle tables against the reference's generated ones: the live library where it is built, and
    always the stored digest of its tables.  The stored-digest check is deliberately the same pin as
    test_oracle_golden.py::test_tables, so that this module's table comparison runs without the library too."""
    w, r, _ = O.port().roots_of_unity(q, n, tw_bits)
    if O.ref_available():
        assert np.array_equal(w, O.ref().table("w", q, n, tw_bits))
        assert np.array_equal(r, O.ref().table("r", q, n, tw_bits))
    # the generated tables as tests/golden/make_golden.py stored them from the library: SHA-256 of w | r, first entries
    G = O.golden("golden_v1")
    assert hashlib.sha256(w.astype("<i4").tobytes() + r.astype("<i4").tobytes()).digest() == G["tab_%d_%d_sha" % (q, n)].tobytes()
    assert [int(w[1]), int(r[0]), int(r[1])] == list(G["tab_%d_%d_head" % (q, n)])


@needs_ref
@pytest.mark.parametrize("q,n,tw", PARAMS)
@pytest.mark.parametrize("op", [O.OP_FWD, O.OP_INV, O.OP_FWD_LARGE, O.OP_INV_LARGE, O.OP_FFT, O.OP_FFT_LARGE,
                                O.OP_NORMALIZE, O.OP_CENTER, O.OP_FLIP, O.OP_MODN, O.OP_SQRN])
def test_unary_ops(q, n, tw, op):
    rng = np.random.default_rng(1000 * op + n + q % 97)
    w, r = O.tables(q, n, tw)
    for variant in variants_for(q):
        for kind in ("uniform", "small", "lazy", "signed"):
            a = rand_inputs(rng, kind, q, (6, n))
            got = O.port().ntt_batch(variant, op, n, q, tw, a, None, w, r)
            exp = O.ref().ntt_batch(variant, op, n, q, tw, a, None, w, r)
            assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], kind)


@needs_ref
@pytest.mark.parametrize("q,n,tw", PARAMS)
@pytest.mark.parametrize("op", [O.OP_PW, O.OP_MULN, O.OP_POLYMUL])
def test_binary_ops(q, n, tw, op):
    rng = np.random.default_rng(77 * op + n)
    w, r = O.tables(q, n, tw)
    for variant in variants_for(q):
        for ka, kb in (("uniform", "uniform"), ("lazy", "uniform"), ("lazy", "lazy"), ("small", "signed")):
            a = rand_inputs(rng, ka, q, (5, n))
            b = rand_inputs(rng, kb, q, (5, n))
            got = O.port().ntt_batch(variant, op, n, q, tw, a, b, w, r)
            exp = O.ref().ntt_batch(variant, op, n, q, tw, a, b, w, r)
            assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], ka, kb)


@needs_ref
@pytest.mark.parametrize("q,n", [(12289, 512), (12289, 1024), (7681, 256)])
def test_pointwise16_and_triple(q, n):
    rng = np.random.default_rng(n)
    w, r = O.tables(q, n, 16)
    key = rng.integers(0, q, size=n).astype(np.int16)
    keys = rng.integers(0, q, size=(4, n)).astype(np.int16)
    for variant in variants_for(q):
        for kind in ("uniform", "small", "lazy"):
            a = rand_inputs(rng, kind, q, (4, n))
            for op in (O.OP_PW16, O.OP_TRIPLE16):
                for b in (key, keys):
                    got = O.port().ntt_batch(variant, op, n, q, 16, a, b, w, r)
                    exp = O.ref().ntt_batch(variant, op, n, q, 16, a, b, w, r)
                    assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], kind, op)


@needs_ref
@pytest.mark.parametrize("q,n,tw", PARAMS)
def test_invert_div_pwr(q, n, tw):
    rng = np.random.default_rng(5)
    for variant in variants_for(q):
        a = rand_inputs(rng, "uniform", q, (3, n))
        a[a == 0] = 1
        a[2, n // 2] = 0                  # row 2 fails half way through and keeps the rest untouched
        b = rand_inputs(rng, "uniform", q, (3, n))
        for op, bb in ((O.OP_INVERT, None), (O.OP_DIV, a), (O.OP_PWR, rng.integers(0, 2 * q, size=(3, n)).astype(np.int32))):
            aa = b if op == O.OP_DIV else a
            got = O.port().ntt_batch(variant, op, n, q, tw, aa, bb, None, None, want_rc=True)
            exp = O.ref().ntt_batch(variant, op, n, q, tw, aa, bb, None, None, want_rc=True)
            assert np.array_equal(got[0], exp[0]) and np.array_equal(got[1], exp[1]) and got[2] == exp[2]
            if op != O.OP_PWR:
                assert list(exp[1]) == [0, 0, 1]


@needs_ref
def test_scalar_and_sparse():
    q, n = 12289, 512
    rng = np.random.default_rng(9)
    a = rand_inputs(rng, "signed", q, (4, n))
    for c in (1, -5, 12288, 77777):
        got = O.port().ntt_batch(O.REFERENCE, O.OP_SCALAR, n, q, 16, a, scalar=c)
        exp = O.ref().ntt_batch(O.REFERENCE, O.OP_SCALAR, n, q, 16, a, scalar=c)
        assert np.array_equal(got, exp)
    omega = 19
    idx = np.stack([rng.choice(n, size=omega, replace=False) for _ in range(4)]).astype(np.int32)
    got = O.port().ntt_batch(O.REFERENCE, O.OP_SPARSE32, n, q, 16, a, idx, scalar=omega)
    exp = O.ref().ntt_batch(O.REFERENCE, O.OP_SPARSE32, n, q, 16, a, idx, scalar=omega)
    assert np.array_equal(got, exp)
    a16 = a.astype(np.int16)
    got = O.port().ntt_batch(O.REFERENCE, O.OP_SPARSE16, n, q, 16, a16, idx, scalar=omega, a_dtype=np.int16)
    exp = O.ref().ntt_batch(O.REFERENCE, O.OP_SPARSE16, n, q, 16, a16, idx, scalar=omega, a_dtype=np.int16)
    assert np.array_equal(got, exp)


@needs_ref
def test_extreme_inputs():
    """Values far outside what schemes pass: wrap-around behaviour must still agree."""
    q, n = 12289, 512
    w, r = O.tables(q, n, 16)
    rng = np.random.default_rng(3)
    a = rng.integers(-2**31, 2**31, size=(8, n), dtype=np.int64).astype(np.int32)
    a[0, :8] = [2**31 - 1, -2**31, -1, 0, 1, q, -q, q * q - 1]
    b = rng.integers(-2**31, 2**31, size=(8, n), dtype=np.int64).astype(np.int32)
    for variant in (O.REFERENCE, O.BARRETT, O.FP, O.AVX):
        for op in (O.OP_MODN, O.OP_NORMALIZE, O.OP_FWD, O.OP_INV, O.OP_PW, O.OP_MULN, O.OP_SQRN, O.OP_POLYMUL):
            if variant == O.REFERENCE and op == O.OP_CENTER:
                continue
            got = O.port().ntt_batch(variant, op, n, q, 16, a, b, w, r)
            exp = O.ref().ntt_batch(variant, op, n, q, 16, a, b, w, r)
            assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], op)


# ---- PRNG / samplers -------------------------------------------------------------------------

def seed_bytes(i, length=64):
    return bytes(((i * 131 + j * 7 + 3) & 0xFF) for j in range(length))


@needs_ref
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_prng_word_stream(prng):
    for s in range(3):
        got = O.port().prng_words(prng, seed_bytes(s), 10000)
        exp = O.ref().prng_words(prng, seed_bytes(s), 10000)
        assert np.array_equal(got, exp)


@needs_ref
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_prng_reseed_boundary(prng):
    """Small seed period: ChaCha reseeds every 64 B of output (rounded to calls), the DRBG clamps to
    4096 updates; draw enough to cross several pool refills and (for ChaCha) many reseeds."""
    got = O.port().prng_words(prng, seed_bytes(7, 48), 3 * 4096 + 5, seed_period=64)
    exp = O.ref().prng_words(prng, seed_bytes(7, 48), 3 * 4096 + 5, seed_period=64)
    assert np.array_equal(got, exp)


@needs_ref
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_prng_mixed_draws(prng):
    rng = np.random.default_rng(11)
    kinds = rng.choice([32, 64, 8, 1, 0], size=3000)
    script = [(int(k), int(rng.integers(1, 32))) for k in kinds]
    got = O.port().prng_script(prng, seed_bytes(1), script)
    exp = O.ref().prng_script(prng, seed_bytes(1), script)
    assert np.array_equal(got, exp)


@needs_ref
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
def test_prng_full_front_end(prng):
    """prng_128 / prng_16 / prng_float / prng_double / prng_mem / prng_reset (DRBG only: reset_chacha20 frees the
    generator, chacha20_csprng.c:58-67) and the byte counters, randomly interleaved with the word and bit draws:
    prng_mem bypasses the 4096-word pool (prng.c:1050-1105), prng_reset keeps the DRBG's stale 1 KiB buffer."""
    rng = np.random.default_rng(5 + prng)
    for trial in range(12):
        seed = rng.integers(0, 256, size=int(rng.integers(36, 80))).astype(np.uint8)
        script = []
        for _ in range(400):
            k = int(rng.choice([32, 64, 8, 1, 16, 0, 128, 2, 3, 4, 4, 6] + ([5] if prng == O.PRNG_AES_CTR_DRBG else [])))
            arg = int(rng.integers(1, 33)) if k == 0 else int(rng.choice([1, 7, 64, 65, 512, 1000, 4096])) if k == 4 else 0
            script.append((k, arg))
        period = int(rng.choice([0, 64, 4096, 0x10000]))
        got = O.port().prng_script(prng, seed, script, period)
        exp = O.ref().prng_script(prng, seed, script, period)
        assert np.array_equal(got, exp), trial


@needs_ref
@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("tail,sigma", [(13.42, 215.0), (13.0, 4.5), (13.42, 19.53), (10.0, 107.0)])
def test_cdf_tables(precision, tail, sigma):
    for blinding in (O.NORMAL_SAMPLES, O.BLINDING_SAMPLES):
        got = O.port().cdf_table(precision, blinding, tail, sigma)
        exp = O.ref().cdf_table(precision, blinding, tail, sigma)
        assert np.array_equal(got, exp)
        # unit_sampling.c:194-210: monotone, first entry 0, last entry all-ones
        assert exp[0] == 0 and exp[-1] == np.iinfo(exp.dtype).max and np.all(np.diff(exp.astype(object)) >= 0)


@needs_ref
@pytest.mark.parametrize("tail,sigma", [(13.42, 215.0), (13.0, 4.5)])
def test_ky_and_bernoulli_tables(tail, sigma):
    for bw in (32, 64):
        got, gb = O.port().ky_table(bw, tail, sigma)
        exp, eb = O.ref().ky_table(bw, tail, sigma)
        assert gb == eb and np.array_equal(got, exp)
    got = O.port().ber_table(tail, sigma)
    exp = O.ref().ber_table(tail, sigma)
    assert got[1:] == exp[1:] and np.array_equal(got[0], exp[0])


@needs_ref
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("blinding", [O.NORMAL_SAMPLES, O.BLINDING_SAMPLES, O.SHUFFLE_SAMPLES])
@pytest.mark.parametrize("precision", [32, 64])
def test_cdf_vectors(prng, blinding, precision):
    seeds = np.array([list(seed_bytes(i)) for i in range(6)], dtype=np.uint8)
    for discard in (0, 2, 6):
        got = O.port().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, 512,
                                     discard=discard, centre=3, calls=2)
        exp = O.ref().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, 512,
                                    discard=discard, centre=3, calls=2)
        assert np.array_equal(got, exp)
    # lengths that are not a power of two: blinding_sample_vector_32 ends with a v[i] <-> v[i & (n-1)] swap pass
    for n in (77, 300, 1):
        got = O.port().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, n, centre=-1, calls=2)
        exp = O.ref().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, n, centre=-1, calls=2)
        assert np.array_equal(got, exp), n


@needs_ref
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("precision", [128, 192])
def test_high_precision_cdf_sampling(prng, precision):
    """gaussian_cdf_sample_128/192 over (a) the table the compiled reference builds itself and (b) an exact
    table written over it; the port restates only the sampling (compare_ge_prec as written)."""
    seeds = np.array([list(seed_bytes(i)) for i in range(5)], dtype=np.uint8)
    own = O.ref().cdf_table(precision, 0, 13.42, 215.0)
    O.port().set_high_table(precision, own)
    got = O.port().gauss_streams(O.SAMPLER_CDF, precision, 0, prng, 13.42, 215.0, seeds, 300)
    assert np.array_equal(got, O.ref().gauss_streams(O.SAMPLER_CDF, precision, 0, prng, 13.42, 215.0, seeds, 300))
    for blinding in (O.NORMAL_SAMPLES, O.BLINDING_SAMPLES, O.SHUFFLE_SAMPLES):
        tab = O.high_precision_cdf_table(precision, 13.42, 215.0, blinding)
        O.ref().set_high_table(precision, tab)
        O.port().set_high_table(precision, tab)
        try:
            for discard in (0, 4):
                got = O.port().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, 300,
                                             discard=discard, centre=-2, calls=2)
                exp = O.ref().gauss_streams(O.SAMPLER_CDF, precision, blinding, prng, 13.42, 215.0, seeds, 300,
                                            discard=discard, centre=-2, calls=2)
                assert np.array_equal(got, exp)
                if blinding == O.NORMAL_SAMPLES and discard == 0:
                    assert 190 < got.std() < 240          # a sane Gaussian, unlike the reference's own table
        finally:
            O.ref().set_high_table(precision, None)


def test_survey_anchor_samples():
    """SURVEY.md 8c anchors (samples of the compiled reference): seed bytes (i*7+3)&0xFF, CDF-64, tail 13.42, sigma 215."""
    ent = np.array([[(i * 7 + 3) & 0xFF for i in range(64)]], dtype=np.uint8)
    for chk in [O.port()] + ([O.ref()] if O.ref_available() else []):
        c = chk.gauss_streams(O.SAMPLER_CDF, 64, 0, O.PRNG_CHACHA, 13.42, 215.0, ent, 12)[0]
        a = chk.gauss_streams(O.SAMPLER_CDF, 64, 0, O.PRNG_AES_CTR_DRBG, 13.42, 215.0, ent, 12)[0]
        assert list(c) == [0, 0, -251, 248, 113, 96, -138, 17, -341, 64, -399, -212]
        assert list(a) == [-319, 333, 125, -307, -208, 85, -140, -269, -1, 74, -120, 180]


@needs_ref
@pytest.mark.parametrize("sampler,precision", [(O.SAMPLER_KNUTH_YAO, 64), (O.SAMPLER_KNUTH_YAO, 32),
                                               (O.SAMPLER_BERNOULLI, 64)])
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("tail,sigma,n", [(13.42, 215.0, 64), (13.0, 4.5, 512)])
def test_ky_bernoulli_samples(sampler, precision, prng, tail, sigma, n):
    seeds = np.array([list(seed_bytes(i)) for i in range(3)], dtype=np.uint8)
    got = O.port().gauss_streams(sampler, precision, 0, prng, tail, sigma, seeds, n)
    exp = O.ref().gauss_streams(sampler, precision, 0, prng, tail, sigma, seeds, n)
    assert np.array_equal(got, exp)
