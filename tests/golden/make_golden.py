"""Generate tests/golden/*.npz from the COMPILED REFERENCE (oracle/_ref/libscref.so).

Needs the reference's source tree, named by REF as for oracle/Makefile (`make -C oracle ref` builds
the library from it; src/unit/unit_ntt.c::test_ibe holds the fixed vectors read below):

    REF=<reference sources> python tests/golden/make_golden.py

The fixtures are what pins the oracle port (and, through it, the CUDA path) on machines where
the reference library is absent.  Inputs are stored next to outputs, so the tests need no RNG
compatibility.
"""
import hashlib
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import _oracle as O  # noqa: E402

REF_SRC = os.environ.get("REF", "")


def variants_for(q):
    v = [O.REFERENCE, O.BARRETT, O.FP, O.AVX]
    if q == 7681:
        v.append(O.SOLINAS_7681)
    if q == 8380417:
        v.append(O.SOLINAS_8380417)
    return v


def main():
    if not os.path.isdir(os.path.join(REF_SRC, "src")):
        sys.exit("make_golden.py: set REF to the reference's source tree")
    ref = O.ref()
    rng = np.random.default_rng(20261017)
    out = {}

    # ---- twiddle tables: digest of every generated table + the first entries ------------------
    for tw, q, n in O.TABLE_PARAMS:
        w = ref.table("w", q, n, tw)
        r = ref.table("r", q, n, tw)
        out["tab_%d_%d_sha" % (q, n)] = np.frombuffer(
            hashlib.sha256(w.astype("<i4").tobytes() + r.astype("<i4").tobytes()).digest(), dtype=np.uint8)
        out["tab_%d_%d_head" % (q, n)] = np.array([w[1], r[0], r[1]], dtype=np.int64)

    # ---- NTT surface ------------------------------------------------------------------------
    params = [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32)]
    unary = [O.OP_FWD, O.OP_INV, O.OP_FWD_LARGE, O.OP_INV_LARGE, O.OP_FFT, O.OP_NORMALIZE, O.OP_CENTER, O.OP_MODN]
    for q, n, tw in params:
        w = ref.table("w", q, n, tw)
        r = ref.table("r", q, n, tw)
        a = np.stack([rng.integers(0, q, n), rng.integers(-300, 301, n), rng.integers(-70000, 600 * q, n)]).astype(np.int32)
        b = np.stack([rng.integers(0, q, n), rng.integers(0, q, n), rng.integers(-q + 1, q, n)]).astype(np.int32)
        key = rng.integers(0, q, n).astype(np.int16)
        tag = "ntt_%d_%d" % (q, n)
        out[tag + "_a"], out[tag + "_b"], out[tag + "_key"] = a, b, key
        for v in variants_for(q):
            for op in unary:
                out["%s_v%d_op%d" % (tag, v, op)] = ref.ntt_batch(v, op, n, q, tw, a, None, w, r)
            for op in (O.OP_PW, O.OP_POLYMUL, O.OP_MULN):
                out["%s_v%d_op%d" % (tag, v, op)] = ref.ntt_batch(v, op, n, q, tw, a, b, w, r)
            if tw == 16:
                for op in (O.OP_PW16, O.OP_TRIPLE16):
                    out["%s_v%d_op%d" % (tag, v, op)] = ref.ntt_batch(v, op, n, q, tw, a, key, w, r)
            nz = a.copy()
            nz[nz % q == 0] = 1
            out["%s_v%d_op%d" % (tag, v, O.OP_INVERT)] = ref.ntt_batch(v, O.OP_INVERT, n, q, tw, nz[:1], None, w, r)

    # ---- the one fixed-vector fixture of the reference: unit_ntt.c test_ibe (:1773-1906) ----
    src = open(os.path.join(REF_SRC, "src/unit/unit_ntt.c")).read()
    body = src[src.index("START_TEST(test_ibe)"):]
    for name in ("g", "f", "c", "s1", "s2"):
        m = re.search(r"SINT32 %s\[512\] = \{([^}]*)\}" % name, body)
        out["ibe_" + name] = np.array([int(x) for x in m.group(1).split(",") if x.strip()], dtype=np.int32)

    # ---- PRNG word streams ----------------------------------------------------------------------
    seed = bytes(((i * 7 + 3) & 0xFF) for i in range(64))
    out["prng_seed"] = np.frombuffer(seed, dtype=np.uint8)
    for name, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
        out["prng_%s_words" % name] = ref.prng_words(pt, seed, 4096 + 64)
        script = [(int(k), int(a)) for k, a in zip(rng.choice([32, 64, 8, 1, 0], 400), rng.integers(1, 32, 400))]
        out["prng_%s_script" % name] = np.array(script, dtype=np.int32)
        out["prng_%s_script_out" % name] = ref.prng_script(pt, seed, script)

    # ---- sampler tables and samples -------------------------------------------------------------
    for prec in (32, 64):
        for bl in (0, 1):
            t = ref.cdf_table(prec, bl, 13.42, 215.0)
            out["cdf%d_b%d_sigma215" % (prec, bl)] = t
    out["cdf64_b0_sigma4p5"] = ref.cdf_table(64, 0, 13.0, 4.5)
    pm, bound = ref.ky_table(64, 13.0, 4.5)
    out["ky64_sigma4p5"] = np.packbits(pm, axis=1)
    out["ky64_sigma4p5_dims"] = np.array([pm.shape[0], pm.shape[1], bound])
    pm, bound = ref.ky_table(64, 13.42, 215.0)
    out["ky64_sigma215_sha"] = np.frombuffer(hashlib.sha256(pm.tobytes()).digest(), dtype=np.uint8)
    out["ky64_sigma215_dims"] = np.array([pm.shape[0], pm.shape[1], bound])
    tab, maxval, maxlog = ref.ber_table(13.42, 215.0)
    out["ber_sigma215"] = tab
    out["ber_sigma215_dims"] = np.array([maxval, maxlog])
    seeds = np.array([[(s * 131 + j * 7 + 3) & 0xFF for j in range(64)] for s in range(4)], dtype=np.uint8)
    out["gauss_seeds"] = seeds
    for pname, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
        for bl in (0, 1, 2):
            for prec in (32, 64):
                out["gauss_cdf%d_%s_b%d" % (prec, pname, bl)] = ref.gauss_streams(
                    O.SAMPLER_CDF, prec, bl, pt, 13.42, 215.0, seeds, 512, calls=2)
        out["gauss_cdf64_%s_discard" % pname] = ref.gauss_streams(
            O.SAMPLER_CDF, 64, 0, pt, 13.42, 215.0, seeds, 512, discard=4)
        out["gauss_ky64_%s" % pname] = ref.gauss_streams(O.SAMPLER_KNUTH_YAO, 64, 0, pt, 13.42, 215.0, seeds, 128)
        out["gauss_ky64s_%s" % pname] = ref.gauss_streams(O.SAMPLER_KNUTH_YAO, 64, 0, pt, 13.0, 4.5, seeds, 512)
        out["gauss_ber64_%s" % pname] = ref.gauss_streams(O.SAMPLER_BERNOULLI, 64, 0, pt, 13.42, 215.0, seeds, 128)
        out["gauss_ber64s_%s" % pname] = ref.gauss_streams(O.SAMPLER_BERNOULLI, 64, 0, pt, 13.0, 4.5, seeds, 512)

    # many variants return identical arrays: each is stored once (O.golden() restores the aliases), which keeps the
    # file under 1 MB
    path = os.path.join(HERE, "golden_v1.npz")
    np.savez_compressed(path, **O.dedup_arrays(out))
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")

    # ---- golden_v2: 128 / 192-bit CDF sampling (gaussian_cdf.c:112-509) over an injected table ------------
    # The table construction needs the reference's multi-precision floats (degenerate under
    # USE_SAFECRYPTO_FLOAT_MP: every entry {2, 2, ..}); the fixture pins the SAMPLING of the compiled reference
    # over (a) the table it builds itself and (b) the exact table of _oracle.high_precision_cdf_table.
    out2 = {"gauss_seeds": seeds}
    for prec in (128, 192):
        own = ref.cdf_table(prec, 0, 13.0, 4.5)
        out2["cdf%d_own_sigma4p5" % prec] = own
        for bl in (0, 1, 2):
            tab = O.high_precision_cdf_table(prec, 13.0, 4.5, bl)
            out2["cdf%d_b%d_sigma4p5" % (prec, bl)] = tab
            ref.set_high_table(prec, tab)
            for pname, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
                out2["gauss_cdf%d_%s_b%d" % (prec, pname, bl)] = ref.gauss_streams(
                    O.SAMPLER_CDF, prec, bl, pt, 13.0, 4.5, seeds, 256, calls=2, discard=(2 if bl == 2 else 0))
            ref.set_high_table(prec, None)
        for pname, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
            out2["gauss_cdf%d_%s_own" % (prec, pname)] = ref.gauss_streams(O.SAMPLER_CDF, prec, 0, pt, 13.0, 4.5, seeds, 64)
    path = os.path.join(HERE, "golden_v2.npz")
    np.savez_compressed(path, **out2)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out2), "arrays")

    # ---- golden_v3 (round 2): the PRNG front end beyond the word stream, module products with a CSPRNG matrix,
    # Knuth-Yao 128 ---------------------------------------------------------------------------------------------
    out3 = {}
    rng = np.random.default_rng(20261017)
    rp_seeds = rng.integers(0, 256, size=(6, 32)).astype(np.uint8)
    out3["rp_seeds"] = rp_seeds
    for name, (q, n, tw, k, l, q_bits) in (("kyber3", (7681, 256, 16, 3, 3, 13)), ("dil", (8380417, 256, 32, 5, 4, 23))):
        y = rng.integers(-4, 5, size=(6, l, n)).astype(np.int32)
        out3["rp_y_%s" % name] = y
        w, r = O.tables(q, n, tw)
        for pname, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
            out3["rp_t_%s_%s" % (name, pname)] = ref.rand_product(tw, O.REFERENCE, n, q, q_bits, k, l, False, pt, rp_seeds, y, w, r)
            if tw == 16:
                out3["rp_tT_%s_%s" % (name, pname)] = ref.rand_product(tw, O.REFERENCE, n, q, q_bits, k, l, True, pt, rp_seeds, y, w, r)
    script = []
    for i in range(300):
        kind = int(rng.choice([32, 64, 8, 1, 16, 0, 128, 2, 3, 4, 4, 6, 5]))
        arg = int(rng.integers(1, 33)) if kind == 0 else int(rng.choice([1, 7, 64, 65, 512, 1000, 4096])) if kind == 4 else 0
        script.append((kind, arg))
    out3["prng_script"] = np.array(script, dtype=np.int32)
    out3["prng_script_seed"] = rng.integers(0, 256, size=48).astype(np.uint8)
    out3["prng_script_aes"] = ref.prng_script(O.PRNG_AES_CTR_DRBG, out3["prng_script_seed"], script, 4096)
    noreset = [(k, a) for k, a in script if k != 5]
    out3["prng_script_chacha"] = ref.prng_script(O.PRNG_CHACHA, out3["prng_script_seed"], noreset, 4096)
    for pname, pt in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
        out3["gauss_ky128_%s" % pname] = ref.gauss_streams(O.SAMPLER_KNUTH_YAO, 128, 0, pt, 13.0, 19.53, seeds, 96)
    path = os.path.join(HERE, "golden_v3.npz")
    np.savez_compressed(path, **out3)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out3), "arrays")


if __name__ == "__main__":
    main()
