"""Parity of the CUDA NTT path (through the C-ABI of libscgpu.so) with the CPU oracle.

Every comparison is bit-exact (integer work).  The oracle is oracle/libscoracle.so (the port,
pinned to the reference in test_oracle_vs_ref.py / test_oracle_golden.py); where the compiled
reference itself travelled to the box (oracle/_ref/libscref.so) it is checked as well.
"""
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
PARAMS = [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32), (8399873, 512, 32)]
DEV = "cuda:0"


def variants_for(q):
    v = [O.REFERENCE, O.BARRETT, O.FP, O.AVX]
    if q == 7681:
        v.append(O.SOLINAS_7681)
    if q == 8380417:
        v.append(O.SOLINAS_8380417)
    return v


def checkers():
    return [O.port()] + ([O.ref()] if O.ref_available() else [])


_plans = {}


def plan(q, n, tw, variant):
    key = (q, n, tw, variant)
    if key not in _plans:
        w, r = O.tables(q, n, tw)
        _plans[key] = (sc.NttPlan(n, q, variant, w, r), w, r)
    return _plans[key]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def run_gpu(q, n, tw, variant, op, a, b=None, scalar=0, inplace=False):
    p, _, _ = plan(q, n, tw, variant)
    da = dev(a.reshape(-1, n) if a.dtype != np.int16 else a.reshape(-1, n))
    db = dev(b) if b is not None else None
    out = da if inplace else torch.full((da.shape[0], n), -7, dtype=torch.int32, device=DEV)
    rc = torch.full((da.shape[0],), -1, dtype=torch.int32, device=DEV)
    p.batch(op, out, da, db, scalar=scalar, rc=rc)
    torch.cuda.synchronize()
    return out.cpu().numpy(), rc.cpu().numpy()


def rand_inputs(rng, kind, q, shape):
    if kind == "uniform":
        return rng.integers(0, q, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "small":
        return rng.integers(-300, 301, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "lazy":
        return rng.integers(-70000, q * 600, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "signed":
        return rng.integers(-q + 1, q, size=shape, dtype=np.int64).astype(np.int32)
    if kind == "extreme":
        x = rng.integers(-2**31, 2**31, size=shape, dtype=np.int64).astype(np.int32)
        x.flat[:8] = [2**31 - 1, -2**31, -1, 0, 1, q, -q, 2**31 - 2]
        return x
    raise ValueError(kind)


UNARY = [O.OP_FWD, O.OP_INV, O.OP_FWD_LARGE, O.OP_INV_LARGE, O.OP_FFT, O.OP_FFT_LARGE, O.OP_NORMALIZE,
         O.OP_CENTER, O.OP_FLIP, O.OP_MODN, O.OP_SQRN]


@pytest.mark.parametrize("q,n,tw", PARAMS)
def test_exact_unary_ops(q, n, tw):
    rng = np.random.default_rng(q + n)
    w, r = O.tables(q, n, tw)
    for variant in variants_for(q):
        for kind in ("uniform", "small", "lazy", "signed", "extreme"):
            a = rand_inputs(rng, kind, q, (37, n))
            for op in UNARY:
                if kind == "extreme" and op == O.OP_CENTER and variant in (O.SOLINAS_7681, O.SOLINAS_8380417):
                    continue
                got, _ = run_gpu(q, n, tw, variant, op, a)
                for chk in checkers():
                    exp = chk.ntt_batch(variant, op, n, q, tw, a, None, w, r)
                    assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], kind, op, chk.prefix)


@pytest.mark.parametrize("q,n,tw", PARAMS)
def test_exact_binary_ops(q, n, tw):
    rng = np.random.default_rng(7 * q + n)
    w, r = O.tables(q, n, tw)
    for variant in variants_for(q):
        for ka, kb in (("uniform", "uniform"), ("lazy", "uniform"), ("lazy", "lazy"), ("small", "signed"), ("extreme", "extreme")):
            a = rand_inputs(rng, ka, q, (21, n))
            b = rand_inputs(rng, kb, q, (21, n))
            for op in (O.OP_PW, O.OP_MULN, O.OP_POLYMUL):
                got, _ = run_gpu(q, n, tw, variant, op, a, b)
                for chk in checkers():
                    exp = chk.ntt_batch(variant, op, n, q, tw, a, b, w, r)
                    assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], ka, kb, op, chk.prefix)
            # shared second operand (b_stride == 0)
            got, _ = run_gpu(q, n, tw, variant, O.OP_PW, a, b[0])
            exp = O.port().ntt_batch(variant, O.OP_PW, n, q, tw, a, b[0], w, r)
            assert np.array_equal(got, exp)


@pytest.mark.parametrize("q,n", [(12289, 512), (12289, 1024), (7681, 256)])
def test_exact_pointwise16_and_triple(q, n):
    rng = np.random.default_rng(n)
    w, r = O.tables(q, n, 16)
    key = rng.integers(0, q, size=n).astype(np.int16)
    keys = rng.integers(0, q, size=(9, n)).astype(np.int16)
    for variant in variants_for(q):
        for kind in ("uniform", "small", "lazy", "extreme"):
            a = rand_inputs(rng, kind, q, (9, n))
            for op in (O.OP_PW16, O.OP_TRIPLE16):
                for b in (key, keys):
                    got, _ = run_gpu(q, n, 16, variant, op, a, b)
                    for chk in checkers():
                        exp = chk.ntt_batch(variant, op, n, q, 16, a, b, w, r)
                        assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], kind, op, chk.prefix)


@pytest.mark.parametrize("q,n,tw", PARAMS)
def test_invert_div_pwr(q, n, tw):
    rng = np.random.default_rng(5)
    for variant in variants_for(q):
        a = rand_inputs(rng, "uniform", q, (5, n))
        a[a == 0] = 1
        a[2, n // 2] = 0
        a[4, 0] = 0
        b = rand_inputs(rng, "uniform", q, (5, n))
        e = rng.integers(0, 2 * q, size=(5, n)).astype(np.int32)
        for op, aa, bb in ((O.OP_INVERT, a, None), (O.OP_DIV, b, a), (O.OP_PWR, a, e)):
            got, rc = run_gpu(q, n, tw, variant, op, aa, bb)
            exp, erc, _ = O.port().ntt_batch(variant, op, n, q, tw, aa, bb, None, None, want_rc=True)
            assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], op)
            if op != O.OP_PWR:
                assert list(rc) == list(erc) == [0, 0, 1, 0, 1]


def test_scalar_sparse_and_inplace():
    q, n, tw = 12289, 512, 16
    rng = np.random.default_rng(9)
    w, r = O.tables(q, n, tw)
    a = rand_inputs(rng, "signed", q, (6, n))
    for c in (1, -5, 12288, 77777):
        got, _ = run_gpu(q, n, tw, O.REFERENCE, O.OP_SCALAR, a, scalar=c)
        assert np.array_equal(got, O.port().ntt_batch(O.REFERENCE, O.OP_SCALAR, n, q, tw, a, scalar=c))
    omega = 19
    idx = np.stack([rng.choice(n, size=omega, replace=False) for _ in range(6)]).astype(np.int32)
    got, _ = run_gpu(q, n, tw, O.REFERENCE, O.OP_SPARSE32, a, idx, scalar=omega)
    assert np.array_equal(got, O.port().ntt_batch(O.REFERENCE, O.OP_SPARSE32, n, q, tw, a, idx, scalar=omega))
    a16 = a.astype(np.int16)
    got, _ = run_gpu(q, n, tw, O.REFERENCE, O.OP_SPARSE16, a16, idx, scalar=omega)
    assert np.array_equal(got, O.port().ntt_batch(O.REFERENCE, O.OP_SPARSE16, n, q, tw, a16, idx, scalar=omega, a_dtype=np.int16))
    # v == t aliasing, as the reference allows (ntt_template.c.in:1570-1576)
    for op in (O.OP_FWD, O.OP_INV, O.OP_NORMALIZE, O.OP_FLIP):
        got, _ = run_gpu(q, n, tw, O.FP, op, a, inplace=True)
        assert np.array_equal(got, O.port().ntt_batch(O.FP, op, n, q, tw, a, None, w, r))


@pytest.mark.parametrize("q,n,tw", [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32)])
def test_golden_vectors_on_gpu(q, n, tw):
    """The committed fixtures generated from the compiled reference, replayed on the GPU."""
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
                got, _ = run_gpu(q, n, tw, v, op, nz[:1])
            elif op in (O.OP_PW16, O.OP_TRIPLE16):
                got, _ = run_gpu(q, n, tw, v, op, a, key)
            elif op in (O.OP_PW, O.OP_POLYMUL, O.OP_MULN):
                got, _ = run_gpu(q, n, tw, v, op, a, b)
            else:
                got, _ = run_gpu(q, n, tw, v, op, a)
            assert np.array_equal(got, G[name]), name
            checked += 1
    assert checked >= 40


def test_ibe_fixture_on_gpu():
    """unit_ntt.c:1773-1906 through the GPU: (s1 - c) f + s2 g == 0 mod 8399873."""
    n, q, v = 512, 8399873, O.FP
    f, g, c, s1, s2 = (G["ibe_" + k].reshape(1, n) for k in ("f", "g", "c", "s1", "s2"))
    s1 = (s1 - c).astype(np.int32)
    run = lambda op, x, y=None: run_gpu(q, n, 32, v, op, x, y)[0]  # noqa: E731
    p1 = run(O.OP_INV_LARGE, run(O.OP_PW, run(O.OP_FWD_LARGE, s1), run(O.OP_FWD, f)))
    p2 = run(O.OP_INV_LARGE, run(O.OP_PW, run(O.OP_FWD_LARGE, s2), run(O.OP_FWD, g)))
    assert not np.any(run(O.OP_NORMALIZE, (p1 + p2).astype(np.int32)))


# ---- fused kernels ------------------------------------------------------------------------------------

FAST_PARAMS = [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32), (18433, 512, 16), (8399873, 512, 32)]


@pytest.fixture(params=["auto", "montgomery", "barrett32", "fq8", "shoup"])
def arithmetic(request):
    """Run the fused-kernel tests with the automatic choice (float-quotient products for small q, warp-local
    32-coefficient schedule), with 32-bit Barrett where applicable, with Montgomery forced for every modulus,
    with the float-quotient arithmetic on the 8-coefficient schedule, and with Shoup products on the warp-local
    schedule for every modulus."""
    old = sc.lib().scgpu_set_fast_arith({"auto": 0, "montgomery": 1, "barrett32": 2, "fq8": 3, "shoup": 4}[request.param])
    yield request.param
    sc.lib().scgpu_set_fast_arith(old)


@pytest.mark.parametrize("q,n,tw", FAST_PARAMS)
def test_fused_polymul_matches_reference_composition(q, n, tw, arithmetic):
    rng = np.random.default_rng(q * 3 + n)
    w, r = O.tables(q, n, tw)
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    for ka, kb, rows in (("uniform", "uniform", 1), ("uniform", "uniform", 1031), ("small", "uniform", 64),
                         ("lazy", "lazy", 64), ("extreme", "extreme", 257), ("signed", "small", 3)):
        a = rand_inputs(rng, ka, q, (rows, n))
        b = rand_inputs(rng, kb, q, (rows, n))
        out = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
        p.polymul(out, dev(a), dev(b))
        torch.cuda.synchronize()
        got = out.cpu().numpy()
        exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, b, w, r)
        assert np.array_equal(got, exp), (ka, kb, rows)
        assert got.min() >= 0 and got.max() < q
        if ka == "uniform" and q < (1 << 15):
            for v in (O.FP, O.AVX):    # canonical output: every sane variant agrees (SURVEY 8a rule 1)
                assert np.array_equal(got[:8], O.port().ntt_batch(v, O.OP_POLYMUL, n, q, tw, a[:8], b[:8], w, r))
    # shared second operand
    a = rand_inputs(rng, "uniform", q, (33, n))
    b = rand_inputs(rng, "uniform", q, (n,))
    out = torch.empty((33, n), dtype=torch.int32, device=DEV)
    p.polymul(out, dev(a), dev(b))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, np.tile(b, (33, 1)), w, r))
    # ... and on a batch large enough for the shared-operand route of the float-quotient policy (one canonical forward
    # transform of b, then the residue-table key product), with any SINT32 in the shared row
    for kb in ("uniform", "signed", "extreme"):
        a = rand_inputs(rng, "lazy" if kb == "extreme" else "uniform", q, (257, n))
        b = rand_inputs(rng, kb, q, (n,))
        out = torch.empty((257, n), dtype=torch.int32, device=DEV)
        p.polymul(out, dev(a), dev(b))
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, np.tile(b, (257, 1)), w, r)), kb


def test_fused_polymul_is_schoolbook_product():
    q, n = 12289, 512
    a, b = G["ntt_12289_512_a"][:1], G["ntt_12289_512_b"][:1]
    p, _, _ = plan(q, n, 16, O.REFERENCE)
    out = torch.empty((1, n), dtype=torch.int32, device=DEV)
    p.polymul(out, dev(a), dev(b))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), G["ntt_12289_512_v0_op%d" % O.OP_POLYMUL][:1])


@pytest.mark.parametrize("q,n", [(12289, 512), (12289, 1024), (7681, 256)])
def test_fused_key_product_matches_triple(q, n, arithmetic):
    rng = np.random.default_rng(n + 1)
    w, r = O.tables(q, n, 16)
    p, _, _ = plan(q, n, 16, O.REFERENCE)
    key = rng.integers(0, q, size=n).astype(np.int16)
    keys = rng.integers(0, q, size=(65, n)).astype(np.int16)
    for kind in ("small", "uniform", "extreme"):
        t = rand_inputs(rng, kind, q, (65, n))
        for k in (key, keys):
            out = torch.empty((65, n), dtype=torch.int32, device=DEV)
            p.mul_key(out, dev(t), dev(k))
            torch.cuda.synchronize()
            exp = O.port().ntt_batch(O.REFERENCE, O.OP_TRIPLE16, n, q, 16, t, k, w, r)
            assert np.array_equal(out.cpu().numpy(), exp), kind
            out32 = torch.empty((65, n), dtype=torch.int32, device=DEV)
            p.mul_key(out32, dev(t), dev(k.astype(np.int32)))
            torch.cuda.synchronize()
            assert np.array_equal(out32.cpu().numpy(), exp)


@pytest.mark.parametrize("q,n,tw", FAST_PARAMS)
def test_canonical_single_transforms(q, n, tw, arithmetic):
    """scgpu_ntt_canonical_batch: forward = normalize_32(fwd_ntt(a)) for every SINT32 input, inverse = inv_ntt(a)
    for inputs the reference itself handles without overflow; and inverse(forward(a)) == a mod q."""
    rng = np.random.default_rng(q + 5 * n)
    w, r = O.tables(q, n, tw)
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    P = O.port()
    for kind, rows in (("uniform", 1), ("uniform", 517), ("small", 33), ("lazy", 64), ("extreme", 65), ("signed", 7)):
        a = rand_inputs(rng, kind, q, (rows, n))
        out = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
        p.ntt_canonical(out, dev(a))
        torch.cuda.synchronize()
        exp = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, n, q, tw, P.ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, a, None, w, r))
        assert np.array_equal(out.cpu().numpy(), exp), ("fwd", kind, rows)
        back = torch.empty_like(out)
        p.ntt_canonical(back, out, inverse=True)
        torch.cuda.synchronize()
        assert np.array_equal(back.cpu().numpy(), np.mod(a.astype(np.int64), q).astype(np.int32)), ("round trip", kind)
    for x in (rng.integers(0, q, size=(129, n)), rng.integers(-q + 1, q, size=(33, n)),
              rng.integers(-(2**31 // n) + 1, 2**31 // n, size=(65, n))):
        x = x.astype(np.int32)
        out = torch.empty((x.shape[0], n), dtype=torch.int32, device=DEV)
        p.ntt_canonical(out, dev(x), inverse=True)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), P.ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, x, None, w, r)), "inv"


@pytest.mark.parametrize("q,n,tw", [(12289, 512, 16), (7681, 256, 16), (8380417, 256, 32)])
def test_fused_key_product_with_arbitrary_32bit_keys(q, n, tw, arithmetic):
    """SINT32 keys far outside [0, q) (the out-of-range path of the key load): against the reference composition
    fwd_ntt, mul_32_pointwise, inv_ntt evaluated by the port."""
    rng = np.random.default_rng(q + n + 7)
    w, r = O.tables(q, n, tw)
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    P = O.port()
    t = rand_inputs(rng, "uniform", q, (40, n))
    for key in (rng.integers(-2**31, 2**31, size=(40, n)).astype(np.int32),
                np.full((40, n), 2**31 - 1, dtype=np.int32), np.full((40, n), -2**31, dtype=np.int32),
                (rng.integers(-4 * q, 4 * q + 1, size=(40, n))).astype(np.int32)):
        out = torch.empty((40, n), dtype=torch.int32, device=DEV)
        p.mul_key(out, dev(t), dev(key))
        torch.cuda.synchronize()
        sh = P.ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, t, None, w, r)
        pr = P.ntt_batch(O.REFERENCE, O.OP_PW, n, q, tw, sh, key, w, r)
        exp = P.ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, pr, None, w, r)
        assert np.array_equal(out.cpu().numpy(), exp)


@pytest.mark.parametrize("q,tw,k,eta", [(7681, 16, 2, 5), (7681, 16, 3, 4), (7681, 16, 4, 3), (8380417, 32, 4, 5)])
def test_matvec_matches_reference_composition(q, tw, k, eta, arithmetic):
    """create_rand_product_32 (module_lwe.c:588-748) with A given in the NTT domain:
    t_i = normalize(inv_ntt(sum_j A_ij o fwd_ntt(s_j)))."""
    n, l, count = 256, k, 19
    rng = np.random.default_rng(k)
    w, r = O.tables(q, n, tw)
    A = rng.integers(0, q, size=(count, k, l, n)).astype(np.int32)
    s = rng.integers(-eta, eta + 1, size=(count, l, n)).astype(np.int32)
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    out = torch.empty((count, k, n), dtype=torch.int32, device=DEV)
    p.matvec(out, dev(A), dev(s), k, l)
    torch.cuda.synchronize()
    P = O.port()
    sh = P.ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, s.reshape(-1, n), None, w, r).reshape(count, l, n)
    exp = np.zeros((count, k, n), dtype=np.int32)
    for i in range(k):
        acc = np.zeros((count, n), dtype=np.int64)
        for j in range(l):
            acc += P.ntt_batch(O.REFERENCE, O.OP_PW, n, q, tw, A[:, i, j], sh[:, j])
        t = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, n, q, tw, acc.astype(np.int32))
        t = P.ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, t, None, w, r)
        exp[:, i] = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, n, q, tw, t)
    assert np.array_equal(out.cpu().numpy(), exp)


def test_full_size_properties():
    """BASELINE config C2 at full size (2^20 polynomials): size-independent properties.
    (1) a * 1 == a mod q; (2) linearity: (a + a') * b == a*b + a'*b mod q; (3) commutativity;
    (4) x^(n-1) * x == -1: negacyclic wrap; (5) the whole output against per-chunk runs; (6) all 2^20 rows against the
    compiled reference."""
    q, n, B = 12289, 512, 1 << 20
    p, _, _ = plan(q, n, 16, O.REFERENCE)
    g = torch.Generator(device=DEV).manual_seed(1)
    a = torch.randint(0, q, (B, n), dtype=torch.int32, device=DEV, generator=g)
    b = torch.randint(0, q, (B, n), dtype=torch.int32, device=DEV, generator=g)
    one = torch.zeros(n, dtype=torch.int32, device=DEV)
    one[0] = 1
    out = torch.empty_like(a)
    p.polymul(out, a, one)
    assert torch.equal(out, a)
    ab = torch.empty_like(a)
    p.polymul(ab, a, b)
    ba = torch.empty_like(a)
    p.polymul(ba, b, a)
    assert torch.equal(ab, ba)
    a2 = torch.randint(0, q, (B, n), dtype=torch.int32, device=DEV, generator=g)
    p.polymul(out, a2, b)
    lhs = torch.empty_like(a)
    p.polymul(lhs, a + a2, b)
    assert torch.equal(lhs, (ab + out) % q)
    del a2, lhs, ba
    xn1 = torch.zeros(n, dtype=torch.int32, device=DEV)
    xn1[n - 1] = 1
    x1 = torch.zeros((4, n), dtype=torch.int32, device=DEV)
    x1[:, 1] = 1
    o4 = torch.empty_like(x1)
    p.polymul(o4, x1, xn1)
    assert int(o4[0, 0]) == q - 1 and int(o4[0, 1:].abs().sum()) == 0
    # chunked re-run must give the same bits as the single launch
    chk = torch.empty((4096, n), dtype=torch.int32, device=DEV)
    for start in (0, 123456, B - 4096):
        p.polymul(chk, a[start:start + 4096], b[start:start + 4096])
        assert torch.equal(chk, ab[start:start + 4096])
    # and EVERY row against the checker: the compiled reference's own fwd, fwd, pointwise, inv over all host threads
    # (a few seconds for 2^20 pairs); the port on a slice when libscref is not available
    w, r = O.tables(q, n, 16)
    if O.ref_available():
        exp = O.ref().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, 16, a.cpu().numpy(), b.cpu().numpy(), w, r, threads=os.cpu_count() or 1)
        assert np.array_equal(ab.cpu().numpy(), exp)
        del exp
    sl = slice(777, 777 + 64)
    exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, 16, a[sl].cpu().numpy(), b[sl].cpu().numpy(), w, r)
    assert np.array_equal(ab[sl].cpu().numpy(), exp)


@pytest.mark.parametrize("q,n,tw,logb", [(12289, 1024, 16, 19), (7681, 256, 16, 20), (8380417, 256, 32, 20)])
def test_full_size_properties_other_shapes(q, n, tw, logb):
    """The other BASELINE shapes (Falcon-1024, Kyber, Dilithium moduli) at full batch size: identity,
    commutativity, linearity, negacyclic wrap, and a slice against the oracle."""
    B = 1 << logb
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    g = torch.Generator(device=DEV).manual_seed(q + n)
    a = torch.randint(0, q, (B, n), dtype=torch.int32, device=DEV, generator=g)
    b = torch.randint(0, q, (B, n), dtype=torch.int32, device=DEV, generator=g)
    one = torch.zeros(n, dtype=torch.int32, device=DEV)
    one[0] = 1
    out = torch.empty_like(a)
    p.polymul(out, a, one)
    assert torch.equal(out, a)
    ab = torch.empty_like(a)
    p.polymul(ab, a, b)
    p.polymul(out, b, a)
    assert torch.equal(ab, out)
    out.copy_(a)
    p.polymul(out, out, b)                          # in place at full concurrency
    assert torch.equal(ab, out)
    a2 = torch.randint(0, q, (B, n), dtype=torch.int32, device=DEV, generator=g)
    p.polymul(out, a2, b)
    lhs = torch.empty_like(a)
    p.polymul(lhs, a + a2, b)                       # inputs up to 2q - 2: lazily reduced operands
    assert torch.equal(lhs, ((ab.long() + out.long()) % q).int())
    xn1 = torch.zeros(n, dtype=torch.int32, device=DEV)
    xn1[n - 1] = 1
    x1 = torch.zeros((4, n), dtype=torch.int32, device=DEV)
    x1[:, 1] = 1
    o4 = torch.empty_like(x1)
    p.polymul(o4, x1, xn1)
    assert int(o4[0, 0]) == q - 1 and int(o4[0, 1:].abs().sum()) == 0
    w, r = O.tables(q, n, tw)
    sl = slice(B - 40, B)
    exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a[sl].cpu().numpy(), b[sl].cpu().numpy(), w, r)
    assert np.array_equal(ab[sl].cpu().numpy(), exp)


@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (8380417, 32, 5, 4)])
def test_full_size_matvec_properties(q, tw, k, l):
    """Module mat-vec at 2^16 instances: A = identity (the constant 1 is the all-ones vector in the NTT domain)
    returns the normalised s; linearity in s; a slice against the oracle composition."""
    n, B = 256, 1 << 16
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    g = torch.Generator(device=DEV).manual_seed(q + k)
    s1 = torch.randint(-5, 6, (B, l, n), dtype=torch.int32, device=DEV, generator=g)
    s2 = torch.randint(0, q, (B, l, n), dtype=torch.int32, device=DEV, generator=g)
    kk = min(k, l)
    eye = torch.zeros((B, kk, l, n), dtype=torch.int32, device=DEV)
    for i in range(kk):
        eye[:, i, i, :] = 1
    out = torch.empty((B, kk, n), dtype=torch.int32, device=DEV)
    p.matvec(out, eye.view(B, kk * l, n), s1, kk, l)
    assert torch.equal(out, s1[:, :kk] % q)
    A = torch.randint(0, q, (B, k * l, n), dtype=torch.int32, device=DEV, generator=g)
    t1 = torch.empty((B, k, n), dtype=torch.int32, device=DEV)
    t2 = torch.empty_like(t1)
    t12 = torch.empty_like(t1)
    p.matvec(t1, A, s1, k, l)
    p.matvec(t2, A, s2, k, l)
    p.matvec(t12, A, s1 + s2, k, l)
    assert torch.equal(t12, ((t1.long() + t2.long()) % q).int())
    assert int(t1.min()) >= 0 and int(t1.max()) < q


def test_small_modulus_inputs_at_the_proof_boundary(arithmetic):
    """Inputs just inside / outside the +-4q window the 32-bit kernels are proven for, adversarial sign
    patterns, and keys at the SINT16 extremes."""
    q, n = 12289, 512
    w, r = O.tables(q, n, 16)
    p, _, _ = plan(q, n, 16, O.REFERENCE)
    rng = np.random.default_rng(12)
    cases = []
    for mag in (4 * q, 4 * q + 1, 4 * q - 1, q - 1, 2**31 - 1):
        cases.append(np.full((3, n), mag, dtype=np.int64))
        cases.append(np.full((3, n), -mag, dtype=np.int64))
        cases.append(mag * rng.choice([-1, 1], size=(3, n)))
    cases.append(np.full((3, n), -2**31, dtype=np.int64))
    for a in cases:
        a = a.astype(np.int32)
        for b in (a, np.ascontiguousarray(a[::-1]), rng.integers(0, q, size=a.shape).astype(np.int32)):
            out = torch.empty((a.shape[0], n), dtype=torch.int32, device=DEV)
            p.polymul(out, dev(a), dev(b))
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, 16, a, b, w, r))
        for kval in (32767, -32768, q - 1, 0):
            key = np.full(n, kval, dtype=np.int16)
            out = torch.empty((a.shape[0], n), dtype=torch.int32, device=DEV)
            p.mul_key(out, dev(a), dev(key))
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_TRIPLE16, n, q, 16, a, key, w, r))


@pytest.mark.parametrize("q,n", [(12289, 512), (12289, 1024), (7681, 256)])
def test_unaligned_rows_take_the_plain_load_path(q, n):
    """The warp-local kernel stages operand rows with bulk copies (TMA), which need 16-byte aligned rows; rows
    at any other alignment go through the LDG variant of the same kernel and must give the same bits.  Also
    ragged counts around the polynomials-per-CTA granularity."""
    w, r = O.tables(q, n, 16)
    p, _, _ = plan(q, n, 16, O.REFERENCE)
    rng = np.random.default_rng(q + n)
    for rows in (1, 7, 33, 161):
        a = rand_inputs(rng, "uniform", q, (rows, n))
        b = rand_inputs(rng, "signed", q, (rows, n))
        exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, 16, a, b, w, r)
        for off_a, off_b in ((0, 0), (1, 0), (0, 3), (2, 1)):
            da = torch.zeros(rows * n + 8, dtype=torch.int32, device=DEV)
            db = torch.zeros(rows * n + 8, dtype=torch.int32, device=DEV)
            da[off_a:off_a + rows * n] = dev(a).reshape(-1)
            db[off_b:off_b + rows * n] = dev(b).reshape(-1)
            out = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
            p.polymul(out, da[off_a:off_a + rows * n].view(rows, n), db[off_b:off_b + rows * n].view(rows, n))
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), exp), (rows, off_a, off_b)
        # in place (v == t aliasing is allowed by the reference, ntt_template.c.in:1570-1576): the prefetch of
        # the next rows must never see a row that has already been overwritten
        ia, ib = dev(a), dev(b)
        p.polymul(ia, ia, ib)
        torch.cuda.synchronize()
        assert np.array_equal(ia.cpu().numpy(), exp), ("in place", rows)
        ia = dev(a)
        p.polymul(ib, ia, ib)
        torch.cuda.synchronize()
        assert np.array_equal(ib.cpu().numpy(), exp), ("in place (second operand)", rows)


def test_host_pipeline_and_ragged_counts():
    q, n, tw = 12289, 512, 16
    w, r = O.tables(q, n, tw)
    rng = np.random.default_rng(3)
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    for rows in (0, 1, 5, 8191, 20000):
        a = rand_inputs(rng, "uniform", q, (rows, n))
        b = rand_inputs(rng, "uniform", q, (rows, n))
        out = np.full((rows, n), -7, dtype=np.int32)
        p.polymul_host(out, a, b, count=rows)
        if rows:
            exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, b, w, r)
            assert np.array_equal(out, exp)
    a = rand_inputs(rng, "uniform", q, (20000, n))
    fwd, back = np.empty_like(a), np.empty_like(a)
    p.ntt_canonical_host(fwd, a)
    p.ntt_canonical_host(back, fwd, inverse=True)
    assert np.array_equal(back, a)
    assert np.array_equal(fwd[:16], O.port().ntt_batch(O.REFERENCE, O.OP_NORMALIZE, n, q, tw,
                                                      O.port().ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, a[:16], None, w, r)))
    a = rand_inputs(rng, "lazy", q, (9000, n))
    out = np.empty_like(a)
    pf, _, _ = plan(q, n, tw, O.FP)
    pf.batch_host(O.OP_FWD, out, a)
    assert np.array_equal(out, O.port().ntt_batch(O.FP, O.OP_FWD, n, q, tw, a, None, w, r))
    rcs = np.full(9000, -1, dtype=np.int32)
    a[a % q == 0] = 1
    a[17, 3] = 0
    pf.batch_host(O.OP_INVERT, out, a, rc=rcs)
    assert rcs[17] == 1 and rcs.sum() == 1


@pytest.mark.parametrize("q,n,tw", [(12289, 512, 16), (12289, 1024, 16), (7681, 256, 16), (8380417, 256, 32)])
def test_work_counter_batches_beyond_one_grid(q, n, tw):
    """Batches larger than one grid-full take their groups from the global work counter (warp32.cuh: claim_next):
    whole output against the oracle, against the static stride (SCGPU_STATIC_SCHED=1), ragged count, and two
    launches in flight on different streams (different counter slots)."""
    rng = np.random.default_rng(n + q)
    rows = 30011
    w, r = O.tables(q, n, tw)
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    P = O.port()
    a, b = rand_inputs(rng, "uniform", q, (rows, n)), rand_inputs(rng, "signed", q, (rows, n))
    da, db = dev(a), dev(b)
    out = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
    p.polymul(out, da, db)
    torch.cuda.synchronize()
    exp = P.ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, b, w, r)
    assert np.array_equal(out.cpu().numpy(), exp)
    fwd = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
    p.ntt_canonical(fwd, da)
    inv = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
    p.ntt_canonical(inv, fwd, inverse=True)
    torch.cuda.synchronize()
    assert torch.equal(inv, da)
    exact = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
    p.batch(O.OP_FWD, exact, da)
    os.environ["SCGPU_STATIC_SCHED"] = "1"
    try:
        out_s, fwd_s, exact_s = torch.empty_like(out), torch.empty_like(out), torch.empty_like(out)
        p.polymul(out_s, da, db)
        p.ntt_canonical(fwd_s, da)
        p.batch(O.OP_FWD, exact_s, da)
        torch.cuda.synchronize()
    finally:
        os.environ["SCGPU_STATIC_SCHED"] = "0"
    assert torch.equal(out_s, out) and torch.equal(fwd_s, fwd) and torch.equal(exact_s, exact)
    # two launches in flight at once
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    o1, o2 = torch.full_like(out, -7), torch.full_like(out, -7)
    torch.cuda.synchronize()
    for _ in range(3):
        p.polymul(o1, da, db, stream=s1)
        p.polymul(o2, db, da, stream=s2)
    torch.cuda.synchronize()
    assert torch.equal(o1, out) and torch.equal(o2, out)
    if n == 256:
        k, l = 3, 2
        inst = 9001
        A = rand_inputs(rng, "uniform", q, (inst, k * l, n))
        s = rng.integers(-4, 5, size=(inst, l, n)).astype(np.int32)
        om = torch.full((inst, k, n), -7, dtype=torch.int32, device=DEV)
        p.matvec(om, dev(A), dev(s), k, l)
        os.environ["SCGPU_STATIC_SCHED"] = "1"
        try:
            om_s = torch.empty_like(om)
            p.matvec(om_s, dev(A), dev(s), k, l)
            torch.cuda.synchronize()
        finally:
            os.environ["SCGPU_STATIC_SCHED"] = "0"
        assert torch.equal(om, om_s)
        sh = P.ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, s[:64].reshape(-1, n), None, w, r).reshape(64, l, n)
        for i in range(k):
            acc = np.zeros((64, n), dtype=np.int64)
            for j in range(l):
                acc += P.ntt_batch(O.REFERENCE, O.OP_PW, n, q, tw, A[:64, i * l + j], sh[:, j])
            t = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, n, q, tw, np.mod(acc, q).astype(np.int32))
            t = P.ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, t, None, w, r)
            assert np.array_equal(om[:64, i].cpu().numpy(), P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, n, q, tw, t))


@pytest.mark.parametrize("q,n", [(12289, 512), (12289, 1024), (7681, 256), (12289, 256)])
def test_base_multiplication_and_in_range_flag(q, n):
    """The two-operand product stops its transforms two stages early and multiplies the residues modulo X^4 - zeta
    (fq_arith.cuh: basemul4).  Same bits as the full-length schedule (SCGPU_NO_BASEMUL=1 at plan creation), as the
    oracle, and -- for operands inside the +-4q window the flag promises -- as the kernel without the range vote
    (SCGPU_PLAN_INPUTS_IN_RANGE), at the window's edges and with adversarial sign patterns."""
    w, r = O.tables(q, n, 16)
    p_bm = sc.NttPlan(n, q, O.REFERENCE, w, r)
    os.environ["SCGPU_NO_BASEMUL"] = "1"
    try:
        p_full = sc.NttPlan(n, q, O.REFERENCE, w, r)
    finally:
        del os.environ["SCGPU_NO_BASEMUL"]
    p_flag = sc.NttPlan(n, q, O.REFERENCE, w, r)
    assert p_flag.set_flags(sc.PLAN_INPUTS_IN_RANGE) == 0
    assert p_flag.set_flags(sc.PLAN_INPUTS_IN_RANGE) == sc.PLAN_INPUTS_IN_RANGE
    rng = np.random.default_rng(q + n)
    x0 = 4 * q
    cases = [(rand_inputs(rng, "uniform", q, (1031, n)), rand_inputs(rng, "uniform", q, (1031, n))),
             (rand_inputs(rng, "signed", q, (65, n)), rand_inputs(rng, "small", q, (65, n))),
             (rng.integers(-x0, x0 + 1, size=(257, n)).astype(np.int32), rng.integers(-x0, x0 + 1, size=(257, n)).astype(np.int32)),
             (np.full((3, n), x0, dtype=np.int32), np.full((3, n), -x0, dtype=np.int32)),
             ((x0 * rng.choice([-1, 1], size=(33, n))).astype(np.int32), (x0 * rng.choice([-1, 1], size=(33, n))).astype(np.int32)),
             (np.full((2, n), q - 1, dtype=np.int32), np.full((2, n), q - 1, dtype=np.int32))]
    one_hot = np.zeros((n, n), dtype=np.int32)
    one_hot[np.arange(n), np.arange(n)] = x0                     # x0 * X^i times a dense operand: every zeta is exercised
    cases.append((one_hot, np.full((n, n), -x0, dtype=np.int32)))
    for a, b in cases:
        exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, 16, a, b, w, r)
        for name, p in (("basemul", p_bm), ("full", p_full), ("flag", p_flag)):
            for aligned in (True, False):                        # bulk-copy and plain-load variants of the kernel
                if aligned:
                    da, db = dev(a), dev(b)
                else:
                    fa = torch.zeros(a.size + 1, dtype=torch.int32, device=DEV)
                    fb = torch.zeros(b.size + 1, dtype=torch.int32, device=DEV)
                    fa[1:] = dev(a).flatten(); fb[1:] = dev(b).flatten()
                    da, db = fa[1:].view(a.shape), fb[1:].view(b.shape)
                out = torch.full(a.shape, -7, dtype=torch.int32, device=DEV)
                p.polymul(out, da, db)
                torch.cuda.synchronize()
                assert np.array_equal(out.cpu().numpy(), exp), (name, aligned, a.shape)
    # arbitrary SINT32 operands stay exact without the flag
    a, b = rand_inputs(rng, "extreme", q, (129, n)), rand_inputs(rng, "lazy", q, (129, n))
    exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, 16, a, b, w, r)
    for p in (p_bm, p_full):
        out = torch.empty(a.shape, dtype=torch.int32, device=DEV)
        p.polymul(out, dev(a), dev(b))
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), exp)
    for p in (p_bm, p_full, p_flag):
        p.close()


@pytest.mark.parametrize("q,tw", [(7681, 16), (12289, 16), (8380417, 32)])
def test_in_range_flag_on_key_products_and_matvec(q, tw):
    """SCGPU_PLAN_INPUTS_IN_RANGE also drops the range votes of the key product and of the module mat-vec; for
    operands inside the promised window the flagged plan returns the bits of the default plan (which the tests above
    pin to the oracle), window edges included."""
    n = 256
    w, r = O.tables(q, n, tw)
    p_def, _, _ = plan(q, n, tw, O.REFERENCE)
    p_flag = sc.NttPlan(n, q, O.REFERENCE, w, r)
    p_flag.set_flags(sc.PLAN_INPUTS_IN_RANGE)
    rng = np.random.default_rng(q)
    x0 = 4 * q
    for t in (rand_inputs(rng, "uniform", q, (131, n)), rand_inputs(rng, "signed", q, (131, n)),
              rng.integers(-x0, x0 + 1, size=(131, n)).astype(np.int32), np.full((5, n), -x0, dtype=np.int32)):
        rows = t.shape[0]
        keys = [rng.integers(0, q, size=(rows, n)).astype(np.int32), rng.integers(-x0, x0 + 1, size=n).astype(np.int32)]
        if tw == 16:
            keys.append(rng.integers(-32768, 32768, size=n).astype(np.int16))
        for key in keys:
            o1 = torch.empty((rows, n), dtype=torch.int32, device=DEV)
            o2 = torch.empty((rows, n), dtype=torch.int32, device=DEV)
            p_def.mul_key(o1, dev(t), dev(key))
            p_flag.mul_key(o2, dev(t), dev(key))
            torch.cuda.synchronize()
            assert torch.equal(o1, o2)
            if key.dtype == np.int32 or tw == 16:
                kk = key if key.ndim == 2 else np.tile(key, (rows, 1))
                if key.dtype == np.int16:
                    exp = O.port().ntt_batch(O.REFERENCE, O.OP_TRIPLE16, n, q, tw, t, key, w, r)
                    assert np.array_equal(o2.cpu().numpy(), exp)
    # canonical single transforms: forward of in-window operands, inverse of in-window NTT-domain values
    for t in (rand_inputs(rng, "uniform", q, (259, n)), rng.integers(-x0, x0 + 1, size=(259, n)).astype(np.int32)):
        for inverse in (False, True):
            o1 = torch.empty((259, n), dtype=torch.int32, device=DEV)
            o2 = torch.empty((259, n), dtype=torch.int32, device=DEV)
            p_def.ntt_canonical(o1, dev(t), inverse=inverse)
            p_flag.ntt_canonical(o2, dev(t), inverse=inverse)
            torch.cuda.synchronize()
            assert torch.equal(o1, o2), inverse
    for k, l in ((2, 2), (3, 2), (4, 4)):
        count = 37
        A = rng.integers(0, q, size=(count, k, l, n)).astype(np.int32)
        A[0] = x0
        A[1] = -x0
        s = rng.integers(-x0, x0 + 1, size=(count, l, n)).astype(np.int32)
        s[2:] = rng.integers(-5, 6, size=(count - 2, l, n))
        o1 = torch.empty((count, k, n), dtype=torch.int32, device=DEV)
        o2 = torch.empty((count, k, n), dtype=torch.int32, device=DEV)
        p_def.matvec(o1, dev(A), dev(s), k, l)
        p_flag.matvec(o2, dev(A), dev(s), k, l)
        torch.cuda.synchronize()
        assert torch.equal(o1, o2), (k, l)
    p_flag.close()


@pytest.mark.parametrize("q,n,tw", PARAMS + [(18433, 512, 16), (12289, 256, 16)])
def test_exact_transforms_when_q_divides_the_products(q, n, tw):
    """The warp-local exact kernels evaluate the fp / avx double quotient in integers wherever that is provably the same
    (ntt_exact_w32.cu header): the C remainder unless q divides the product, the canonical residue for the double
    lanes.  The exceptional case is forced here: inputs that are multiples of q (sums of multiples stay multiples, so
    every butterfly of every stage is in the exceptional case), zeros, sparse rows, rows at +-2^29 / +-2^31 (beyond the
    bound of the 32-bit-table form), against the compiled reference and the port, all variants, forward and inverse."""
    rng = np.random.default_rng(q - n)
    w, r = O.tables(q, n, tw)
    kmax = (2**31 - 1) // q
    rows = []
    rows.append(q * rng.integers(-3, 4, size=(9, n)))
    rows.append(q * rng.integers(-kmax, kmax + 1, size=(9, n)))
    rows.append(np.zeros((2, n), dtype=np.int64))
    sparse = np.zeros((6, n), dtype=np.int64)
    sparse[np.arange(6), rng.integers(0, n, size=6)] = [1, -1, q, -q, q * kmax, 12345]
    rows.append(sparse)
    big = rng.choice([2**29, -(2**29), 2**29 - 1, 2**29 + 1, 2**31 - 1, -(2**31)], size=(6, n))
    rows.append(big)
    mixed = rng.integers(0, q, size=(8, n))
    mixed[:, ::3] = q * rng.integers(-5, 6, size=mixed[:, ::3].shape)
    rows.append(mixed)
    a = np.concatenate(rows).astype(np.int32)
    for variant in variants_for(q):
        for op in (O.OP_FWD, O.OP_INV):
            got, _ = run_gpu(q, n, tw, variant, op, a)
            for chk in checkers():
                exp = chk.ntt_batch(variant, op, n, q, tw, a, None, w, r)
                assert np.array_equal(got, exp), (O.VARIANT_NAMES[variant], op, chk.prefix, np.argwhere(got != exp)[:4])


# the remaining moduli of the reference's parameter sets (ENS / DLP 5767169 and 10223617, Ring-TESLA 51750913 -- 26 bits,
# beyond both fused arithmetics --, 4206593, 16813057), 32-bit tables
OTHER_SCHEME_PARAMS = [(5767169, 512), (5767169, 1024), (10223617, 512), (10223617, 1024), (51750913, 512), (51750913, 1024),
                       (4206593, 512), (16813057, 512)]


@pytest.mark.parametrize("q,n", OTHER_SCHEME_PARAMS)
def test_other_scheme_moduli(q, n):
    """Every modulus the reference's schemes use beyond the headline sets: the variant-exact transforms and pointwise
    product of every live variant against the checkers, the fused product / key product against the reference
    composition, the canonical single transforms (which compose the exact kernels where no fused arithmetic serves)."""
    tw = 32
    rng = np.random.default_rng(q % 1000 + n)
    w, r = O.tables(q, n, tw)
    a = rand_inputs(rng, "uniform", q, (37, n))
    b = rand_inputs(rng, "uniform", q, (37, n))
    for v in (O.REFERENCE, O.BARRETT, O.FP, O.AVX):
        for chk in checkers():
            for op, second in ((O.OP_FWD, None), (O.OP_INV, None), (O.OP_PW, b), (O.OP_NORMALIZE, None)):
                got, _ = run_gpu(q, n, tw, v, op, a, second)
                assert np.array_equal(got, chk.ntt_batch(v, op, n, q, tw, a, second, w, r)), (v, op)
        lz = rand_inputs(rng, "lazy", q, (9, n))
        got, _ = run_gpu(q, n, tw, v, O.OP_FWD, lz)
        assert np.array_equal(got, O.port().ntt_batch(v, O.OP_FWD, n, q, tw, lz, None, w, r)), v
    p, _, _ = plan(q, n, tw, O.REFERENCE)
    exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, b, w, r)
    out = torch.full((37, n), -7, dtype=torch.int32, device=DEV)
    p.polymul(out, dev(a), dev(b))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), exp)
    for ka, kb, rows in (("lazy", "lazy", 64), ("extreme", "extreme", 129), ("signed", "small", 5)):
        xa, xb = rand_inputs(rng, ka, q, (rows, n)), rand_inputs(rng, kb, q, (rows, n))
        o2 = torch.full((rows, n), -7, dtype=torch.int32, device=DEV)
        p.polymul(o2, dev(xa), dev(xb))
        torch.cuda.synchronize()
        assert np.array_equal(o2.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, xa, xb, w, r)), (ka, kb)
        # inverse transform: inputs the reference itself handles without overflow (sums of n terms)
        xi = rng.integers(-(2**31 // n) + 1, 2**31 // n, size=(rows, n)).astype(np.int32)
        p.ntt_canonical(o2, dev(xi), inverse=True)
        torch.cuda.synchronize()
        assert np.array_equal(o2.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, xi, None, w, r)), ka
        kx = rand_inputs(rng, kb, q, (n,))
        p.mul_key(o2, dev(xa), dev(kx))
        torch.cuda.synchronize()
        shx = O.port().ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, xa, None, w, r)
        prx = O.port().ntt_batch(O.REFERENCE, O.OP_PW, n, q, tw, shx, np.tile(kx, (rows, 1)), w, r)
        assert np.array_equal(o2.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, prx, None, w, r)), (ka, kb, "key")
    big = rand_inputs(rng, "uniform", q, (20011, n))            # beyond one grid-full: the work counter
    outb = torch.empty((20011, n), dtype=torch.int32, device=DEV)
    p.polymul(outb, dev(big), dev(b[0]))
    torch.cuda.synchronize()
    sel = np.r_[0:5, 20000:20011]
    assert np.array_equal(outb.cpu().numpy()[sel], O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, big[sel], np.tile(b[0], (len(sel), 1)), w, r))
    fwd = torch.empty((37, n), dtype=torch.int32, device=DEV)
    p.ntt_canonical(fwd, dev(a))
    torch.cuda.synchronize()
    assert np.array_equal(fwd.cpu().numpy(), np.mod(O.port().ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, a, None, w, r), q))
    back = torch.empty_like(fwd)
    p.ntt_canonical(back, fwd, inverse=True)
    torch.cuda.synchronize()
    assert np.array_equal(back.cpu().numpy(), a)
    key = rand_inputs(rng, "uniform", q, (n,))
    p.mul_key(out, dev(a), dev(key))
    torch.cuda.synchronize()
    sh = O.port().ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, a, None, w, r)
    pr = O.port().ntt_batch(O.REFERENCE, O.OP_PW, n, q, tw, sh, np.tile(key, (37, 1)), w, r)
    assert np.array_equal(out.cpu().numpy(), O.port().ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, pr, None, w, r))


@pytest.mark.parametrize("q,n", [(8380417, 256), (8399873, 512), (10223617, 1024), (51750913, 512), (51750913, 1024)])
def test_large_modulus_inputs_at_the_proof_boundary(q, n):
    """The Shoup-policy kernels at the edge of their interval analysis (analyse_sh: inputs up to 4 q, every intermediate
    inside the signed 32-bit range -- for the 26-bit modulus the whole of it): constant and adversarially signed rows of
    magnitude 4 q, through the default plan (range vote) and through a plan that declares them in range (no vote)."""
    tw = 32
    w, r = O.tables(q, n, tw)
    rng = np.random.default_rng(q % 97 + n)
    P = O.port()
    checked, flagged = sc.NttPlan(n, q, sc.REFERENCE, w, r), sc.NttPlan(n, q, sc.REFERENCE, w, r)
    flagged.set_flags(sc.PLAN_INPUTS_IN_RANGE)
    cases = []
    for mag in (4 * q, 4 * q - 1, q - 1):
        cases.append(np.full((3, n), mag, dtype=np.int64))
        cases.append(np.full((3, n), -mag, dtype=np.int64))
        cases.append(mag * rng.choice([-1, 1], size=(3, n)))
        alt = np.full((3, n), mag, dtype=np.int64)
        alt[:, 1::2] = -mag
        cases.append(alt)
    for a in cases:
        a = a.astype(np.int32)
        for b in (a, np.ascontiguousarray(a[:, ::-1]), rng.integers(0, q, size=a.shape).astype(np.int32)):
            exp = P.ntt_batch(O.REFERENCE, O.OP_POLYMUL, n, q, tw, a, b, w, r)
            for p in (checked, flagged):
                out = torch.empty((a.shape[0], n), dtype=torch.int32, device=DEV)
                p.polymul(out, dev(a), dev(b))
                torch.cuda.synchronize()
                assert np.array_equal(out.cpu().numpy(), exp)
        key = rng.integers(0, q, size=n).astype(np.int32)
        sh = P.ntt_batch(O.REFERENCE, O.OP_FWD, n, q, tw, a, None, w, r)
        pr = P.ntt_batch(O.REFERENCE, O.OP_PW, n, q, tw, sh, np.tile(key, (a.shape[0], 1)), w, r)
        expk = P.ntt_batch(O.REFERENCE, O.OP_INV, n, q, tw, pr, None, w, r)
        expf = np.mod(sh.astype(np.int64), q).astype(np.int32)
        for p in (checked, flagged):
            out = torch.empty((a.shape[0], n), dtype=torch.int32, device=DEV)
            p.mul_key(out, dev(a), dev(key))
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), expk)
            p.ntt_canonical(out, dev(a))
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), expf)
