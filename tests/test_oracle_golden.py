"""The oracle port against (1) the committed fixtures generated from the compiled reference
(tests/golden/make_golden.py) and (2) the known answers the reference's own tests hold for
this path (src/unit/unit_ntt.c, src/unit/unit_sampling.c, src/unit/crypto/unit_aes.c,
test/functional/func_ntt.c).  Needs neither a GPU nor /root/reference."""
import ctypes
import hashlib
import os

import numpy as np
import pytest

import _oracle as O

G = O.golden("golden_v1")
P = O.port()


def variants_for(q):
    v = [O.REFERENCE, O.BARRETT, O.FP, O.AVX]
    if q == 7681:
        v.append(O.SOLINAS_7681)
    if q == 8380417:
        v.append(O.SOLINAS_8380417)
    return v


# ---- tables -------------------------------------------------------------------------------------

@pytest.mark.parametrize("tw_bits,q,n", O.TABLE_PARAMS)
def test_tables(tw_bits, q, n):
    w, r, g = P.roots_of_unity(q, n, tw_bits)
    sha = hashlib.sha256(w.astype("<i4").tobytes() + r.astype("<i4").tobytes()).digest()
    assert sha == G["tab_%d_%d_sha" % (q, n)].tobytes()
    assert [int(w[1]), int(r[0]), int(r[1])] == list(G["tab_%d_%d_head" % (q, n)])
    assert pow(g, n, q) == q - 1 and (int(r[0]) * n) % q == q - 1


def test_survey_table_anchors():
    # SURVEY.md 8a: g = 49 / 7 / 62 / 1753 ; r[0] = 24 / 30 / 32736
    assert P.roots_of_unity(12289, 512, 16)[2] == 49
    assert P.roots_of_unity(12289, 1024, 16)[2] == 7
    assert P.roots_of_unity(7681, 256, 16)[2] == 62
    assert P.roots_of_unity(8380417, 256, 32)[2] == 1753
    assert P.roots_of_unity(12289, 512, 16)[1][0] == 24
    assert P.roots_of_unity(7681, 256, 16)[1][0] == 30
    assert P.roots_of_unity(8380417, 256, 32)[1][0] == 32736


def test_primitive_roots():
    # unit_ntt.c:1382-1402
    f = P.lib.orc_find_primitive_root
    f.restype = ctypes.c_int64
    f.argtypes = [ctypes.c_int64]
    assert f(7681) == 17 and f(12289) == 11


# ---- scalar KATs of unit_ntt.c ----------------------------------------------------------------------

def test_muln_kats():
    # unit_ntt.c:166-187,322-343: 1234 * 5678 mod 12289 == 1922 in every variant
    for v in (O.REFERENCE, O.BARRETT, O.FP):
        assert P.scalar("muln", v, 512, 12289, 1234, 5678) == 1922
    # unit_ntt.c:189-252: edge cases around q and q^2 (Barrett and fp), written as x * 1
    for v in (O.BARRETT, O.FP):
        assert P.scalar("muln", v, 512, 12289, 1, 12289) == 0
        assert P.scalar("muln", v, 512, 12289, 1, 12290) == 1
        assert P.scalar("muln", v, 512, 12289, 1, 12289 * 12289 - 1) == 12288
        assert P.scalar("muln", v, 512, 12289, 1, 12289 * 12289) == 0
    # unit_ntt.c:254-281: the reference variant keeps the sign of the dividend
    assert P.scalar("muln", O.REFERENCE, 512, 12289, -1234, 5678) == -1922
    assert P.scalar("muln", O.REFERENCE, 512, 12289, 1234, -5678) == -1922
    assert P.scalar("muln", O.REFERENCE, 512, 12289, -1234, -5678) == 1922
    # unit_ntt.c:85-108: q = 7681
    for v in (O.REFERENCE, O.BARRETT, O.FP):
        assert P.scalar("muln", v, 256, 7681, 1234, 5678) == (1234 * 5678) % 7681


def test_fp_equals_reference_on_negative_sweep():
    # unit_ntt.c:283-320: x = -64 i, y = 0x7FFFFFFF for 16384 points
    for i in range(0, 16384, 37):
        x = -64 * i
        assert (P.scalar("muln", O.FP, 512, 12289, x, 0x7FFFFFFF)
                == P.scalar("muln", O.REFERENCE, 512, 12289, x, 0x7FFFFFFF))


def test_modn_sweep():
    # func_ntt.c:70-103 sweeps modn over 0 .. 2^30-1 against a wrap-around counter; sampled here
    n, q = 512, 12289
    x = np.concatenate([np.arange(0, 1 << 16), np.arange((1 << 30) - (1 << 16), 1 << 30),
                        np.random.default_rng(0).integers(0, 1 << 30, 1 << 16)]).astype(np.int32)
    x = x[: (x.size // n) * n].reshape(-1, n)
    for v in (O.REFERENCE, O.BARRETT, O.FP):
        got = P.ntt_batch(v, O.OP_MODN, n, q, 16, x)
        assert np.array_equal(got, x % q)


# ---- transform properties the reference tests assert ---------------------------------------------------

@pytest.mark.parametrize("q,n,tw", [(8399873, 512, 32), (12289, 1024, 16), (12289, 512, 16), (7681, 256, 16)])
def test_ntt_times_inverse_is_one(q, n, tw):
    # unit_ntt.c:554-942: NTT(g) * NTT(g)^-1 -> INTT = (1, 0, ..., 0)
    w, r = O.tables(q, n, tw)
    rng = np.random.default_rng(q + n)
    # Barrett with k = 30 is only congruent, not canonical, for 23-bit moduli (m = 127): the
    # reference tests it on the 13/14-bit moduli only
    for v in ((O.REFERENCE, O.FP) if q > (1 << 15) else (O.REFERENCE, O.BARRETT, O.FP)):
        g = rng.integers(-2, 3, size=(1, n)).astype(np.int32)
        gh = P.ntt_batch(v, O.OP_FWD, n, q, tw, g, None, w, r)
        gh = P.ntt_batch(v, O.OP_NORMALIZE, n, q, tw, gh)
        if np.any(gh == 0):
            continue
        gi, rc, _ = P.ntt_batch(v, O.OP_INVERT, n, q, tw, gh, want_rc=True)
        assert rc[0] == 0
        prod = P.ntt_batch(v, O.OP_PW, n, q, tw, gh, gi)
        one = P.ntt_batch(v, O.OP_INV, n, q, tw, prod, None, w, r)
        assert one[0, 0] == 1 and not np.any(one[0, 1:])


@pytest.mark.parametrize("q,n,tw", [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32)])
def test_fwd_inv_identity(q, n, tw):
    # unit_ntt.c:946-1036,1156-1300
    w, r = O.tables(q, n, tw)
    a = np.random.default_rng(n).integers(0, q, size=(4, n)).astype(np.int32)
    for v in variants_for(q):
        if v == O.BARRETT and q > (1 << 15):
            continue              # k = 30 Barrett is not a working reduction for 23-bit q (SURVEY 8a)
        back = P.ntt_batch(v, O.OP_INV, n, q, tw, P.ntt_batch(v, O.OP_FWD, n, q, tw, a, None, w, r), None, w, r)
        if v in (O.SOLINAS_7681, O.SOLINAS_8380417):
            back = back % q       # Solinas folds are not canonical (SURVEY 8a)
        assert np.array_equal(back % q, a)


def test_ibe_fixture():
    """unit_ntt.c:1773-1906: (s1 - c) * f + s2 * g == 0 mod 8399873 through the large/non-large
    32-bit-table transforms of the floating-point variant -- the only golden polymul in the tree."""
    n, q, v = 512, 8399873, O.FP
    w, r = O.tables(q, n, 32)
    f, g, c, s1, s2 = (G["ibe_" + k].reshape(1, n) for k in ("f", "g", "c", "s1", "s2"))
    s1 = (s1 - c).astype(np.int32)
    s1h = P.ntt_batch(v, O.OP_FWD_LARGE, n, q, 32, s1, None, w, r)
    s2h = P.ntt_batch(v, O.OP_FWD_LARGE, n, q, 32, s2, None, w, r)
    fh = P.ntt_batch(v, O.OP_FWD, n, q, 32, f, None, w, r)
    gh = P.ntt_batch(v, O.OP_FWD, n, q, 32, g, None, w, r)
    p1 = P.ntt_batch(v, O.OP_INV_LARGE, n, q, 32, P.ntt_batch(v, O.OP_PW, n, q, 32, s1h, fh), None, w, r)
    p2 = P.ntt_batch(v, O.OP_INV_LARGE, n, q, 32, P.ntt_batch(v, O.OP_PW, n, q, 32, s2h, gh), None, w, r)
    tot = P.ntt_batch(v, O.OP_NORMALIZE, n, q, 32, (p1 + p2).astype(np.int32))
    assert not np.any(tot)


# ---- golden NTT vectors ---------------------------------------------------------------------------

@pytest.mark.parametrize("q,n,tw", [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32)])
def test_golden_ntt(q, n, tw):
    w, r = O.tables(q, n, tw)
    tag = "ntt_%d_%d" % (q, n)
    a, b, key = G[tag + "_a"], G[tag + "_b"], G[tag + "_key"]
    checked = 0
    for v in variants_for(q):
        for op in range(22):
            name = "%s_v%d_op%d" % (tag, v, op)
            if name not in G:
                continue
            if op == O.OP_INVERT:
                nz = a.copy()
                nz[nz % q == 0] = 1
                got = P.ntt_batch(v, op, n, q, tw, nz[:1], None, w, r)
            elif op in (O.OP_PW16, O.OP_TRIPLE16):
                got = P.ntt_batch(v, op, n, q, tw, a, key, w, r)
            elif op in (O.OP_PW, O.OP_POLYMUL, O.OP_MULN):
                got = P.ntt_batch(v, op, n, q, tw, a, b, w, r)
            else:
                got = P.ntt_batch(v, op, n, q, tw, a, None, w, r)
            assert np.array_equal(got, G[name]), name
            checked += 1
    assert checked >= 40


def test_golden_polymul_is_negacyclic_product():
    """Independent of any NTT: schoolbook product mod (x^n + 1, q) equals the reference-variant
    golden output (and therefore the fp / avx ones, which the fixture shows to be identical)."""
    q, n = 12289, 512
    a, b = G["ntt_12289_512_a"][0].astype(object), G["ntt_12289_512_b"][0].astype(object)
    c = [0] * n
    for i in range(n):
        for j in range(n):
            if i + j < n:
                c[i + j] += a[i] * b[j]
            else:
                c[i + j - n] -= a[i] * b[j]
    c = np.array([int(x) % q for x in c], dtype=np.int32)
    for v in (O.REFERENCE, O.FP, O.AVX):
        assert np.array_equal(G["ntt_12289_512_v%d_op%d" % (v, O.OP_POLYMUL)][0], c)


# ---- PRNG ---------------------------------------------------------------------------------------------

def test_aes256_fips197():
    # FIPS-197 C.3 (the block cipher unit_aes.c:141-189 pins with the SP 800-38A vectors)
    key = bytes(range(32))
    pt = bytes.fromhex("00112233445566778899aabbccddeeff")
    out = (ctypes.c_uint8 * 16)()
    P.lib.orc_aes256_encrypt_block(key, pt, out)
    assert bytes(out).hex() == "8ea2b7ca516745bfeafc49904b496089"
    # SP 800-38A F.5.5 CTR-AES256 block 1 keystream input -> output
    key = bytes.fromhex("603deb1015ca71be2b73aef0857d77811f352c073b6108d72d9810a30914dff4")
    ctr = bytes.fromhex("f0f1f2f3f4f5f6f7f8f9fafbfcfdfeff")
    P.lib.orc_aes256_encrypt_block(key, ctr, out)
    assert bytes(out).hex() == "0bdf7df1591716335e9a8b15c860c502"


@pytest.mark.parametrize("name,pt", [("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)])
def test_golden_prng(name, pt):
    seed = G["prng_seed"].tobytes()
    exp = G["prng_%s_words" % name]
    assert np.array_equal(P.prng_words(pt, seed, exp.size), exp)
    assert np.array_equal(P.prng_script(pt, seed, G["prng_%s_script" % name]), G["prng_%s_script_out" % name])
    if name == "chacha":
        assert not np.any(exp[:3])          # three leading zero words (chacha20_csprng.c:72-84)


# ---- samplers -----------------------------------------------------------------------------------------

def test_golden_sampler_tables():
    for prec in (32, 64):
        for bl in (0, 1):
            t = P.cdf_table(prec, bl, 13.42, 215.0)
            assert np.array_equal(t, G["cdf%d_b%d_sigma215" % (prec, bl)])
            # unit_sampling.c:194-210,292-309
            assert t[0] == 0 and t[-1] == np.iinfo(t.dtype).max and t.size == 4096
    assert np.array_equal(P.cdf_table(64, 0, 13.0, 4.5), G["cdf64_b0_sigma4p5"])
    pm, bound = P.ky_table(64, 13.0, 4.5)
    assert [pm.shape[0], pm.shape[1], bound] == list(G["ky64_sigma4p5_dims"])
    assert np.array_equal(np.packbits(pm, axis=1), G["ky64_sigma4p5"])
    pm, bound = P.ky_table(64, 13.42, 215.0)
    assert [pm.shape[0], pm.shape[1], bound] == list(G["ky64_sigma215_dims"]) == [64, 2887, 2886]
    assert hashlib.sha256(pm.tobytes()).digest() == G["ky64_sigma215_sha"].tobytes()
    tab, maxval, maxlog = P.ber_table(13.42, 215.0)
    assert np.array_equal(tab, G["ber_sigma215"]) and [maxval, maxlog] == list(G["ber_sigma215_dims"]) == [2886, 12]


@pytest.mark.parametrize("pname,pt", [("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)])
def test_golden_samples(pname, pt):
    seeds = G["gauss_seeds"]
    for bl in (0, 1, 2):
        for prec in (32, 64):
            got = P.gauss_streams(O.SAMPLER_CDF, prec, bl, pt, 13.42, 215.0, seeds, 512, calls=2)
            assert np.array_equal(got, G["gauss_cdf%d_%s_b%d" % (prec, pname, bl)])
            # unit_sampling.c:212-216: |sample| < 2^ceil_log2(tail*sigma) (twice that when blinded)
            assert np.abs(got).max() < (8192 if bl == 1 else 4096)
    got = P.gauss_streams(O.SAMPLER_CDF, 64, 0, pt, 13.42, 215.0, seeds, 512, discard=4)
    assert np.array_equal(got, G["gauss_cdf64_%s_discard" % pname])
    for key, smp, tail, sigma, n in (("ky64", O.SAMPLER_KNUTH_YAO, 13.42, 215.0, 128),
                                     ("ky64s", O.SAMPLER_KNUTH_YAO, 13.0, 4.5, 512),
                                     ("ber64", O.SAMPLER_BERNOULLI, 13.42, 215.0, 128),
                                     ("ber64s", O.SAMPLER_BERNOULLI, 13.0, 4.5, 512)):
        got = P.gauss_streams(smp, 64, 0, pt, tail, sigma, seeds, n)
        assert np.array_equal(got, G["gauss_%s_%s" % (key, pname)])


@pytest.mark.parametrize("pname,pt", [("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)])
@pytest.mark.parametrize("precision", [128, 192])
def test_golden_high_precision_samples(pname, pt, precision):
    """golden_v2: samples of the compiled reference's 128 / 192-bit CDF sampler over injected tables."""
    G2 = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v2.npz"))
    seeds = G2["gauss_seeds"]
    P.set_high_table(precision, G2["cdf%d_own_sigma4p5" % precision])
    assert np.array_equal(P.gauss_streams(O.SAMPLER_CDF, precision, 0, pt, 13.0, 4.5, seeds, 64),
                          G2["gauss_cdf%d_%s_own" % (precision, pname)])
    for bl in (0, 1, 2):
        tab = G2["cdf%d_b%d_sigma4p5" % (precision, bl)]
        assert np.array_equal(tab, O.high_precision_cdf_table(precision, 13.0, 4.5, bl))
        P.set_high_table(precision, tab)
        got = P.gauss_streams(O.SAMPLER_CDF, precision, bl, pt, 13.0, 4.5, seeds, 256, calls=2, discard=(2 if bl == 2 else 0))
        assert np.array_equal(got, G2["gauss_cdf%d_%s_b%d" % (precision, pname, bl)])


def test_sample_statistics():
    """func_samplers.c histograms 2^20 samples; here: mean ~ 0 and std ~ sigma for each sampler."""
    seeds = np.random.default_rng(1).integers(0, 256, size=(64, 64)).astype(np.uint8)
    x = P.gauss_streams(O.SAMPLER_CDF, 64, 0, O.PRNG_AES_CTR_DRBG, 13.42, 215.0, seeds, 2048)
    assert abs(x.mean()) < 3.0 and abs(x.std() - 215.0) < 3.0
    x = P.gauss_streams(O.SAMPLER_KNUTH_YAO, 64, 0, O.PRNG_AES_CTR_DRBG, 13.0, 4.5, seeds, 512)
    # the reference's Knuth-Yao walk is not an exact sampler (column 0 carries the full 2/(sigma
    # sqrt(2 pi)) mass and the table pointer drifts after a hit): it measures std ~ 3.9 at sigma 4.5.
    # Bit-exactness with it is what is pinned above; this only guards against gross breakage.
    assert abs(x.mean()) < 0.2 and 3.5 < x.std() < 4.7
    x = P.gauss_streams(O.SAMPLER_BERNOULLI, 64, 0, O.PRNG_AES_CTR_DRBG, 13.0, 4.5, seeds, 256)
    assert abs(x.mean()) < 0.3 and abs(x.std() - 4.5) < 0.3


def test_round2_fixtures_prng_front_end_and_ky128():
    """golden_v3.npz (generated from the compiled reference): prng_128 / float / double / mem / reset / counters in a
    random interleaving, and Knuth-Yao at 128 rows."""
    import os
    G3 = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v3.npz"))
    script = [tuple(int(v) for v in row) for row in G3["prng_script"]]
    seed = G3["prng_script_seed"]
    assert np.array_equal(O.port().prng_script(O.PRNG_AES_CTR_DRBG, seed, script, 4096), G3["prng_script_aes"])
    noreset = [(k, a) for k, a in script if k != 5]
    assert np.array_equal(O.port().prng_script(O.PRNG_CHACHA, seed, noreset, 4096), G3["prng_script_chacha"])
    seeds = np.array([[(s * 131 + j * 7 + 3) & 0xFF for j in range(64)] for s in range(4)], dtype=np.uint8)
    for pname, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
        got = O.port().gauss_streams(O.SAMPLER_KNUTH_YAO, 128, 0, pt, 13.0, 19.53, seeds, 96)
        assert np.array_equal(got, G3["gauss_ky128_%s" % pname])
