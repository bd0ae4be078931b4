"""Module products (scgpu_matvec_batch, scgpu_matvec_shared_batch, scgpu_rand_product_csprng_batch, its _shared_batch
form and both _host twins) against an exact reference, at the input and accumulator limits of include/scgpu.h.

The mat-vec is linear mod q, so for ANY SINT32 input its exact value is

    t_i = G ( sum_j (A_ij mod q) o F (s_j mod q) ) mod q

with F and G the n x n matrices over Z_q of the reference's forward and inverse transforms (the port's OP_FWD / OP_INV
applied to the n unit vectors).  The tests without the gpu mark check that reference itself: G F = I, G (F a o F b) is
the negacyclic product, it agrees with the port's composition normalize(inv(normalize(sum pw(A, fwd(s))))) on benign
inputs, and normalize(fwd(s)) = F (s mod q) for extreme s.  The gpu tests compare every module-product kernel with it:
inputs at and beyond the +-4q window of SCGPU_PLAN_INPUTS_IN_RANGE, l at the largest value each modulus admits, every
arithmetic of scgpu_set_fast_arith, the kernel-selection variables, unaligned rows and batch sizes around grid-fulls."""
import functools
import os

import numpy as np
import pytest

import _oracle as O

try:
    import torch
except ImportError:                                            # the reference checks need numpy only
    torch = None

HAVE_GPU = torch is not None and torch.cuda.is_available()
DEV = "cuda:0"
N = 256
INT32_MIN, INT32_MAX = -2**31, 2**31 - 1


def gpu_test(f):
    return pytest.mark.gpu(pytest.mark.skipif(not HAVE_GPU, reason="no CUDA device")(f))


# ---- the exact reference ---------------------------------------------------------------------------------------------

def mulmod(X, M, q):
    """X @ M mod q, exactly, for X [m, n] and M [n, n] with entries in [0, q), q < 2^23.  The contraction runs in
    column chunks of 16 and is reduced after each chunk: a chunk sums 16 products below 2^46, so every partial sum is an
    integer below 2^50 and the float64 products are exact whatever order the BLAS adds them in."""
    assert q < 2**23 and X.min() >= 0 and X.max() < q and M.min() >= 0 and M.max() < q
    acc = np.zeros((X.shape[0], M.shape[1]), dtype=np.int64)
    Xf, Mf = X.astype(np.float64), M.astype(np.float64)
    for c in range(0, X.shape[1], 16):
        acc = (acc + (Xf[:, c:c + 16] @ Mf[c:c + 16]).astype(np.int64)) % q
    return acc


@functools.lru_cache(maxsize=None)
def transforms(q, tw):
    """(F, G) as row-major maps over Z_q: the transform of a batch of rows X is X @ F mod q (row i of F is OP_FWD of the
    i-th unit vector), the inverse transform is X @ G mod q."""
    w, r = O.tables(q, N, tw)
    eye = np.eye(N, dtype=np.int32)
    P = O.port()
    F = P.ntt_batch(O.REFERENCE, O.OP_FWD, N, q, tw, eye, None, w, r).astype(np.int64) % q
    G = P.ntt_batch(O.REFERENCE, O.OP_INV, N, q, tw, eye, None, w, r).astype(np.int64) % q
    return F, G


def forward(q, tw, s):
    """F (s mod q) for s [..., n] of any SINT32."""
    F, _ = transforms(q, tw)
    return mulmod(s.reshape(-1, N).astype(np.int64) % q, F, q).reshape(s.shape)


def product(q, tw, A, Fs):
    """t [count, k, n] from A ([k, l, n] shared or [count, k, l, n]) and the transformed vectors Fs [count, l, n]."""
    _, G = transforms(q, tw)
    Am = A.astype(np.int64) % q
    count, k = Fs.shape[0], A.shape[-3]
    acc = np.zeros((count, k, N), dtype=np.int64)
    for i in range(k):
        Ai = Am[i] if A.ndim == 3 else Am[:, i]
        acc[:, i] = (Ai * Fs).sum(axis=-2) % q                  # l products below 2^46 each
    return mulmod(acc.reshape(-1, N), G, q).reshape(count, k, N).astype(np.int32)


def exact_matvec(q, tw, A, s):
    return product(q, tw, A, forward(q, tw, s))


def port_composition(q, tw, A, s):
    """normalize(inv_ntt(normalize(sum_j pw(A_ij, fwd_ntt(s_j))))) through the port, A [count, k, l, n]."""
    w, r = O.tables(q, N, tw)
    P = O.port()
    count, k, l = A.shape[0], A.shape[1], A.shape[2]
    sh = P.ntt_batch(O.REFERENCE, O.OP_FWD, N, q, tw, s.reshape(-1, N), None, w, r).reshape(count, l, N)
    exp = np.zeros((count, k, N), dtype=np.int32)
    for i in range(k):
        acc = np.zeros((count, N), dtype=np.int64)
        for j in range(l):
            acc += P.ntt_batch(O.REFERENCE, O.OP_PW, N, q, tw, A[:, i, j], sh[:, j])
        t = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, N, q, tw, acc.astype(np.int32))
        t = P.ntt_batch(O.REFERENCE, O.OP_INV, N, q, tw, t, None, w, r)
        exp[:, i] = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, N, q, tw, t)
    return exp


MODULI = [(7681, 16), (12289, 16), (8380417, 32)]


@pytest.mark.parametrize("q,tw", MODULI)
def test_reference_transforms_invert_each_other(q, tw):
    F, G = transforms(q, tw)
    assert np.array_equal(mulmod(F, G, q), np.eye(N, dtype=np.int64))
    assert np.array_equal(mulmod(G, F, q), np.eye(N, dtype=np.int64))


@pytest.mark.parametrize("q,tw", MODULI)
def test_reference_is_the_negacyclic_product(q, tw):
    """G (F a o F b) against the schoolbook product mod (x^n + 1, q) in Python integers."""
    rng = np.random.default_rng(q)
    _, G = transforms(q, tw)
    for _ in range(2):
        a, b = rng.integers(0, q, size=(2, N))
        got = mulmod(forward(q, tw, a[None]) * forward(q, tw, b[None]) % q, G, q)[0]
        ai, bi = [int(x) for x in a], [int(x) for x in b]
        exp = [0] * N
        for i in range(N):
            for j in range(N):
                if i + j < N:
                    exp[i + j] += ai[i] * bi[j]
                else:
                    exp[i + j - N] -= ai[i] * bi[j]
        assert [int(x) for x in got] == [x % q for x in exp]


@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (12289, 16, 2, 4), (8380417, 32, 6, 5), (8380417, 32, 1, 5)])
def test_reference_equals_the_port_composition(q, tw, k, l):
    """On benign inputs (A in [0, q), |s| <= 5) the formula gives the bits of the port's composition."""
    rng = np.random.default_rng(q + k + l)
    A = rng.integers(0, q, size=(9, k, l, N)).astype(np.int32)
    s = rng.integers(-5, 6, size=(9, l, N)).astype(np.int32)
    assert np.array_equal(exact_matvec(q, tw, A, s), port_composition(q, tw, A, s))


@pytest.mark.parametrize("q,tw", MODULI)
def test_reference_forward_transform_of_extreme_inputs(q, tw):
    """normalize(fwd_ntt(s)) = F (s mod q) for s = +-4q constant, alternating +-4q, random SINT32, INT32_MAX and
    INT32_MIN: the mathematical residue is also the reference library's own result for such inputs."""
    w, r = O.tables(q, N, tw)
    P = O.port()
    rng = np.random.default_rng(q + 1)
    x0 = 4 * q
    alt = np.where(np.arange(N) % 2 == 0, x0, -x0)
    rows = np.stack([np.full(N, x0), np.full(N, -x0), alt, -alt, rng.integers(INT32_MIN, INT32_MAX + 1, size=N),
                     np.full(N, INT32_MAX), np.full(N, INT32_MIN)]).astype(np.int32)
    got = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, N, q, tw, P.ntt_batch(O.REFERENCE, O.OP_FWD, N, q, tw, rows, None, w, r))
    assert np.array_equal(got.astype(np.int64), forward(q, tw, rows))


# ---- inputs ----------------------------------------------------------------------------------------------------------
# In the window |x| <= 4q (both plans) and beyond it (the default plan only: "any SINT32 input is exact").

A_IN = ["uniform", "zero", "q-1", "+4q", "-4q", "+-4q"]
A_OUT = ["+(4q+1)", "-(4q+1)", "sint32"]
S_IN = ["small", "+4q", "-4q", "alt4q", "+-4q", "onehot4q"]
S_OUT = ["+(4q+1)", "-(4q+1)", "+-(4q+1)", "extreme"]
ETA = 5


def sint32(rng, shape):
    x = rng.integers(INT32_MIN, INT32_MAX + 1, size=shape, dtype=np.int64)
    x.flat[:4] = [INT32_MAX, INT32_MIN, INT32_MAX - 1, INT32_MIN + 1]
    return x


def pattern(rng, name, q, shape):
    """One operand of `shape` ([k, l, n] or [l, n]) following the named pattern."""
    x0 = 4 * q
    if name == "uniform":
        x = rng.integers(0, q, size=shape)
    elif name == "zero":
        x = np.zeros(shape, dtype=np.int64)
    elif name == "q-1":
        x = np.full(shape, q - 1)
    elif name == "small":
        x = rng.integers(-ETA, ETA + 1, size=shape)
    elif name in ("+4q", "-4q", "+(4q+1)", "-(4q+1)"):
        x = np.full(shape, {"+4q": x0, "-4q": -x0, "+(4q+1)": x0 + 1, "-(4q+1)": -x0 - 1}[name])
    elif name in ("+-4q", "+-(4q+1)"):
        x = rng.choice(np.array([-1, 1]), size=shape) * (x0 if name == "+-4q" else x0 + 1)
    elif name == "alt4q":
        x = np.broadcast_to(np.where(np.arange(N) % 2 == 0, x0, -x0), shape).copy()
    elif name == "onehot4q":                                  # 4q X^i, i random per row
        x = np.zeros(shape, dtype=np.int64).reshape(-1, N)
        x[np.arange(x.shape[0]), rng.integers(0, N, size=x.shape[0])] = x0
        x = x.reshape(shape)
    elif name == "sint32":
        x = sint32(rng, shape)
    elif name == "extreme":                                    # the extreme pattern of test_gpu_ntt.rand_inputs
        x = rng.integers(INT32_MIN, INT32_MAX + 1, size=shape, dtype=np.int64)
        x.flat[:8] = [INT32_MAX, INT32_MIN, -1, 0, 1, q, -q, INT32_MAX - 1]
    else:
        raise ValueError(name)
    return np.asarray(x, dtype=np.int64).astype(np.int32)


@functools.lru_cache(maxsize=None)
def exact_case(q, tw, k, l):
    """Matrices and vectors of every pattern for one shape, with the exact products of every (matrix, vector) pair:
    ({A name: [k, l, n]}, [s names], s [len, l, n], {A name: t [len, k, n]})."""
    rng = np.random.default_rng(1009 * k + 31 * l + q % 1000)
    A = {a: pattern(rng, a, q, (k, l, N)) for a in A_IN + A_OUT}
    snames = S_IN + S_OUT
    s = np.stack([pattern(rng, n, q, (l, N)) for n in snames])
    Fs = forward(q, tw, s)
    return A, snames, s, {a: product(q, tw, A[a], Fs) for a in A}


def assert_exact(got, exp, label, names=None, index=None):
    """Equal, or a message naming the case, the instance, the output row and the first differing coefficient."""
    if np.array_equal(got, exp):
        return
    bad = np.argwhere(got != exp)
    c, i, j = (int(v) for v in bad[0])
    inst = index[c] if index is not None else c
    what = " (%s)" % names[c] if names is not None else ""
    raise AssertionError("%s: instance %d%s, output row %d, coefficient %d: got %d, expected %d; %d coefficients of %d "
                         "instances differ" % (label, inst, what, i, j, got[c, i, j], exp[c, i, j], len(bad),
                                               len(np.unique(bad[:, 0]))))


# ---- which kernel each case reaches ----------------------------------------------------------------------------------
# route() restates the choice of launch_matvec (ntt_fast.cu) and launch_matvec_w32 (warp32.cuh) for n = 256:
#   arithmetic 1 (Montgomery)                        -> k_matvec
#   arithmetic 2 (Barrett-32): q < 2^20              -> k_matvec_sq, else k_matvec
#   arithmetic 3 (fq8):        q = 7681, 12289       -> k_matvec_fq, else k_matvec
#   arithmetic 4 (Shoup)                             -> the warp-local kernels with ArSh
#   arithmetic 0 (automatic):  q = 7681, 12289       -> the warp-local kernels with ArFq (float quotients)
#                              q = 8380417           -> the warp-local kernels with ArSh
# and among the warp-local kernels:
#   ArFq, l >= SCGPU_MATVEC16_MINL (default 1), s rows 16-byte aligned (A too unless shared), bulk copies allowed
#   (SCGPU_NO_TMA unset), SCGPU_MATVEC_STASH32 unset    -> k_matvec16_w32<CHK, IACC, SHARED_A>, IACC unless
#                                                          SCGPU_MATVEC_FLOAT_ACC (then ArFq::acc_fin's shared float
#                                                          quotient sums the l products)
#   else, the same alignment, 2 <= k <= 8, SCGPU_MATVEC_ONE_WARP unset
#                                                       -> k_matvec_rows_w32<CHK, SHARED_A> (always with bulk copies;
#                                                          with ArFq it also sums through acc_fin)
#   else                                                -> k_matvec_w32<TMA, CHK, SHARED_A>, TMA when A and s rows are
#                                                          aligned and SCGPU_NO_TMA is unset
# CHK (the range vote on the operands) is on for the default plan and off for the SCGPU_PLAN_INPUTS_IN_RANGE plan; with
# SHARED_A the matrix is reduced once by k_matrix_table and only s is voted on.  The warp-local kernels accept l up to
# sh32_mv_lmax (5 for q = 8380417) with ArSh and up to 4 with ArFq; the others up to 4.

def route(q, k, l, arith, flagged, shared, env=(), misalign=None):
    env = dict(env)
    chk = "CHK" if not flagged else "NOCHK"
    sh = ",SHARED_A" if shared else ""
    small = q < 59000
    if arith == 1 or (arith in (2, 3) and not small):
        return "k_matvec%s" % ("<SHARED_A>" if shared else "")
    if arith == 2:
        return "k_matvec_sq%s" % ("<SHARED_A>" if shared else "")
    if arith == 3:
        return "k_matvec_fq%s" % ("<SHARED_A>" if shared else "")
    ar = "ArFq" if (arith == 0 and small) else "ArSh"
    tma_ok = env.get("SCGPU_NO_TMA", "0") == "0"
    tma = tma_ok and misalign not in ("A", "s")
    tma_rows = tma_ok and misalign != "s" if shared else tma
    if (ar == "ArFq" and l >= int(env.get("SCGPU_MATVEC16_MINL", "1")) and tma_rows
            and env.get("SCGPU_MATVEC_STASH32", "0") == "0"):
        iacc = "IACC" if env.get("SCGPU_MATVEC_FLOAT_ACC", "0") == "0" else "FACC"
        return "k_matvec16_w32<ArFq,%s,%s%s>" % (chk, iacc, sh)
    if tma_rows and 2 <= k <= 8 and env.get("SCGPU_MATVEC_ONE_WARP", "0") == "0":
        return "k_matvec_rows_w32<%s,%s%s>" % (ar, chk, sh)
    return "k_matvec_w32<%s,%s,%s%s>" % (ar, "TMA" if tma else "NOTMA", chk, sh)


def lmax(q, arith):
    """Largest l the launcher accepts: 5 for q = 8380417 on the Shoup-policy kernels (automatic or Shoup arithmetic),
    otherwise 4."""
    return 5 if (q == 8380417 and arith in (0, 4)) else 4


ARITHS = [0, 1, 2, 3, 4]
ARITH_IDS = ["auto", "montgomery", "barrett32", "fq8", "shoup"]
SMALL_SHAPES = [(q, 16, k, l) for q in (7681, 12289) for k in range(1, 5) for l in range(1, 5)] + \
               [(7681, 16, 9, 2), (12289, 16, 9, 2)]
DIL_SHAPES = [(8380417, 32, k, l) for k, l in ((5, 4), (6, 5), (1, 5), (8, 1), (9, 5), (12, 3))]
SHAPES = SMALL_SHAPES + DIL_SHAPES

# automatic arithmetic only: (q, tw, k, l, environment, misaligned operand) -- the kernel each reaches is in the id
SELECTION = [
    (7681, 16, 3, 3, {"SCGPU_MATVEC_ONE_WARP": "1"}, None),
    (8380417, 32, 5, 4, {"SCGPU_MATVEC_ONE_WARP": "1"}, None),
    (8380417, 32, 6, 5, {"SCGPU_MATVEC_ONE_WARP": "1"}, None),
    (7681, 16, 3, 3, {"SCGPU_MATVEC_STASH32": "1"}, None),
    (12289, 16, 4, 4, {"SCGPU_MATVEC_STASH32": "1"}, None),
    (7681, 16, 1, 4, {"SCGPU_MATVEC_STASH32": "1"}, None),
    (7681, 16, 9, 2, {"SCGPU_MATVEC_STASH32": "1"}, None),
    (7681, 16, 4, 4, {"SCGPU_MATVEC_STASH32": "1", "SCGPU_MATVEC_ONE_WARP": "1"}, None),
    (7681, 16, 4, 4, {"SCGPU_MATVEC_FLOAT_ACC": "1"}, None),
    (12289, 16, 4, 4, {"SCGPU_MATVEC_FLOAT_ACC": "1"}, None),
    (12289, 16, 1, 4, {"SCGPU_MATVEC_FLOAT_ACC": "1"}, None),
    (7681, 16, 3, 3, {"SCGPU_NO_TMA": "1"}, None),
    (12289, 16, 4, 4, {"SCGPU_NO_TMA": "1"}, None),
    (8380417, 32, 6, 5, {"SCGPU_NO_TMA": "1"}, None),
    (7681, 16, 3, 3, {"SCGPU_MATVEC16_MINL": "4"}, None),
    (12289, 16, 2, 4, {"SCGPU_MATVEC16_MINL": "5"}, None),
    (7681, 16, 1, 3, {"SCGPU_MATVEC16_MINL": "4"}, None),
    (7681, 16, 3, 3, {}, "A"),
    (7681, 16, 3, 3, {}, "s"),
    (12289, 16, 4, 4, {}, "out"),
    (8380417, 32, 5, 4, {}, "A"),
    (8380417, 32, 6, 5, {}, "s"),
    (8380417, 32, 1, 5, {}, "out"),
]

# (q, tw, k, l) of the batch-size test (automatic arithmetic)
BATCH_SHAPES = [(7681, 16, 3, 3), (12289, 16, 2, 4), (8380417, 32, 5, 4), (8380417, 32, 6, 5), (8380417, 32, 1, 5)]

# (q, tw, k, l, q_bits, transposes) of the seeded products
RAND_SHAPES = [(7681, 16, 2, 2, 13, (False, True)), (7681, 16, 3, 3, 13, (False, True)), (7681, 16, 4, 4, 13, (False, True)),
               (12289, 16, 3, 3, 14, (False,)), (8380417, 32, 5, 4, 23, (False,)), (8380417, 32, 6, 5, 23, (False,))]

# the instantiations the module products can reach; every one must be the target of some case below
INSTANTIATIONS = (
    ["k_matvec16_w32<ArFq,%s,%s%s>" % (c, a, s) for c in ("CHK", "NOCHK") for a in ("IACC", "FACC") for s in ("", ",SHARED_A")]
    + ["k_matvec_rows_w32<%s,%s%s>" % (ar, c, s) for ar in ("ArFq", "ArSh") for c in ("CHK", "NOCHK") for s in ("", ",SHARED_A")]
    + ["k_matvec_w32<%s,%s,%s%s>" % (ar, t, c, s) for ar in ("ArFq", "ArSh") for t in ("TMA", "NOTMA")
       for c in ("CHK", "NOCHK") for s in ("", ",SHARED_A")]
    + [kern + s for kern in ("k_matvec", "k_matvec_sq", "k_matvec_fq") for s in ("", "<SHARED_A>")])


def reached():
    """Every instantiation the gpu tests of this module launch."""
    got = set()
    for flagged in (0, 1):
        for shared in (False, True):
            for q, tw, k, l in SHAPES:
                for arith in ARITHS:
                    if l <= lmax(q, arith):
                        got.add(route(q, k, l, arith, flagged, shared))
            for q, tw, k, l, env, mis in SELECTION:
                got.add(route(q, k, l, 0, flagged, shared, env, mis))
    return got


def test_cases_reach_every_instantiation():
    missing = sorted(set(INSTANTIATIONS) - reached())
    assert not missing, missing


# ---- GPU -------------------------------------------------------------------------------------------------------------

if HAVE_GPU:
    import libsafecrypto_b200 as sc
    from libsafecrypto_b200 import binding as B


@pytest.fixture(scope="module")
def plans():
    """(default plan, SCGPU_PLAN_INPUTS_IN_RANGE plan) per modulus, created once for the module."""
    made = {}

    def get(q, tw):
        if (q, tw) not in made:
            w, r = O.tables(q, N, tw)
            p_def = sc.NttPlan(N, q, sc.REFERENCE, w, r)
            p_flag = sc.NttPlan(N, q, sc.REFERENCE, w, r)
            p_flag.set_flags(sc.PLAN_INPUTS_IN_RANGE)
            made[(q, tw)] = (p_def, p_flag)
        return made[(q, tw)]
    yield get
    for p_def, p_flag in made.values():
        p_def.close()
        p_flag.close()


@pytest.fixture(params=ARITHS, ids=ARITH_IDS)
def arith(request):
    old = sc.lib().scgpu_set_fast_arith(request.param)
    yield request.param
    sc.lib().scgpu_set_fast_arith(old)


@pytest.fixture
def auto_arith():
    old = sc.lib().scgpu_set_fast_arith(0)
    yield 0
    sc.lib().scgpu_set_fast_arith(old)


def dev(a, misaligned=False):
    """A device copy of a; misaligned: starting one word after a 16-byte boundary."""
    a = np.ascontiguousarray(a)
    if not misaligned:
        return torch.from_numpy(a).to(DEV)
    buf = torch.empty(a.size + 4, dtype=torch.int32, device=DEV)
    v = buf[1:1 + a.size].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.data_ptr() % 16 == 4
    return v


def out_buffer(count, k, misaligned=False):
    buf = torch.full((count * k * N + 4,), -7, dtype=torch.int32, device=DEV)
    return (buf[1:] if misaligned else buf)[:count * k * N].view(count, k, N)


def run_matvec(p, A, s, k, l, shared, misalign=None):
    o = out_buffer(s.shape[0], k, misalign == "out")
    fn = p.matvec_shared if shared else p.matvec
    fn(o, dev(A, misalign == "A"), dev(s, misalign == "s"), k, l)
    torch.cuda.synchronize()
    return o.cpu().numpy()


def check_patterns(p, flagged, q, tw, k, l, label, arith=0, env=(), misalign=None):
    """Every (matrix, vector) pattern pair through both entry points; the in-range plan gets the in-window pairs only.
    matvec: one call with one pair per instance; matvec_shared: one call per matrix with every vector."""
    A, snames, s, exp = exact_case(q, tw, k, l)
    anames = A_IN if flagged else A_IN + A_OUT
    sidx = [i for i, n in enumerate(snames) if n in S_IN or not flagged]
    pairs = [(a, i) for a in anames for i in sidx]
    got = run_matvec(p, np.stack([A[a] for a, _ in pairs]), s[[i for _, i in pairs]], k, l, False, misalign)
    assert_exact(got, np.stack([exp[a][i] for a, i in pairs]),
                 "%s matvec [%s]" % (label, route(q, k, l, arith, flagged, False, env, misalign)),
                 ["A %s, s %s" % (a, snames[i]) for a, i in pairs])
    for a in anames:
        got = run_matvec(p, A[a], s[sidx], k, l, True, misalign)
        assert_exact(got, exp[a][sidx], "%s matvec_shared A %s [%s]" % (label, a, route(q, k, l, arith, flagged, True, env, misalign)),
                     ["s %s" % snames[i] for i in sidx])


def refused(fn):
    with pytest.raises(sc.ScgpuError):
        fn()


def plan_name(flagged):
    return "in-range" if flagged else "default"


@gpu_test
@pytest.mark.parametrize("q,tw,k,l", SHAPES)
def test_matvec_exact(q, tw, k, l, arith, plans):
    """Both entry points under every arithmetic on both plans, against the exact reference; l above what the arithmetic
    serves must be refused."""
    z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=DEV)  # noqa: E731
    for flagged, p in enumerate(plans(q, tw)):
        if l > lmax(q, arith):
            refused(lambda: p.matvec(z(3, k, N), z(3, k, l, N), z(3, l, N), k, l))
            refused(lambda: p.matvec_shared(z(3, k, N), z(k, l, N), z(3, l, N), k, l))
            continue
        label = "q=%d k=%d l=%d arith=%s %s plan" % (q, k, l, ARITH_IDS[arith], plan_name(flagged))
        check_patterns(p, flagged, q, tw, k, l, label, arith)


@gpu_test
@pytest.mark.parametrize("q,tw,k,l,env,misalign", SELECTION,
                         ids=["%d-%dx%d-%s" % (c[0], c[2], c[3], route(c[0], c[2], c[3], 0, 0, False, c[4], c[5]))
                              + ("-" + "-".join(sorted(c[4])) if c[4] else "") + ("-misaligned-" + c[5] if c[5] else "")
                              for c in SELECTION])
def test_kernel_selection_and_alignment(q, tw, k, l, env, misalign, auto_arith, plans, monkeypatch):
    """The launch-time selection variables and rows one word off a 16-byte boundary, against the exact reference."""
    for var, val in env.items():
        monkeypatch.setenv(var, val)
    for flagged, p in enumerate(plans(q, tw)):
        label = "q=%d k=%d l=%d %s misaligned=%s %s plan" % (q, k, l, env, misalign, plan_name(flagged))
        check_patterns(p, flagged, q, tw, k, l, label, 0, env, misalign)


def grid_instances(q, k, l, shared):
    """Instances in one grid-full of the kernel launch_matvec_w32 picks under the automatic arithmetic."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if q < 59000:                                              # k_matvec16_w32: 4 instances per one-warp CTA
        smem = (4 * (296 + 264) + l * 4 * 168) * 4
        return sms * min(16, (227 * 1024) // (smem + 1088)) * 4
    if 2 <= k <= 8:                                            # k_matvec_rows_w32: 4 instances per CTA of k warps
        smem = (l * 4 * 296 + k * (4 * 296 + (0 if shared else 4 * 264))) * 4
        return sms * max(1, min((227 * 1024) // (smem + 1280), 65536 // (k * 32 * 128))) * 4
    smem = ((l + 1) * 4 * 296 + 4 * 264) * 4                   # k_matvec_w32
    return sms * min(16, (227 * 1024) // (smem + 1088)) * 4


def compared(count, G, rng):
    """The whole batch up to 4096 instances; above: first, last, grid boundaries +-2 and 256 random instances."""
    if count <= 4096:
        return np.arange(count)
    idx = {0, count - 1}
    for b in range(G, count, G):
        idx.update(range(max(0, b - 2), min(count, b + 3)))
    idx.update(int(x) for x in rng.integers(0, count, size=256))
    return np.array(sorted(idx))


@gpu_test
@pytest.mark.parametrize("q,tw,k,l", BATCH_SHAPES)
def test_batch_sizes(q, tw, k, l, auto_arith, plans):
    """1, 3, 4, 5, 37 instances, one grid-full -1 / +0 / +1 and twelve grid-fulls plus a ragged tail, both entry
    points, both plans; operands at random points of the +-4q window and its corners."""
    g = torch.Generator(device=DEV).manual_seed(q + 7 * k + l)
    rng = np.random.default_rng(q + k + l)
    x0 = 4 * q
    G = {shared: grid_instances(q, k, l, shared) for shared in (False, True)}
    counts = {shared: [1, 3, 4, 5, 37, G[shared] - 1, G[shared], G[shared] + 1, 12 * G[shared] + 5] for shared in G}
    top = max(max(c) for c in counts.values())
    signs = lambda *shape: torch.randint(0, 2, shape, dtype=torch.int32, device=DEV, generator=g) * (2 * x0) - x0  # noqa: E731
    s = torch.randint(-x0, x0 + 1, (top, l, N), dtype=torch.int32, device=DEV, generator=g)
    s[::3] = signs(len(range(0, top, 3)), l, N)
    A_sh = signs(k, l, N)
    A = torch.randint(-x0, x0 + 1, (top, k, l, N), dtype=torch.int32, device=DEV, generator=g)
    A[1::3] = signs(len(range(1, top, 3)), k, l, N)
    picks = {(shared, c): compared(c, G[shared], rng) for shared in G for c in counts[shared]}
    need = np.unique(np.concatenate(list(picks.values())))
    pos = np.full(top, -1)
    pos[need] = np.arange(len(need))
    Fs = forward(q, tw, s[torch.from_numpy(need).to(DEV)].cpu().numpy())
    exp = {True: product(q, tw, A_sh.cpu().numpy(), Fs),
           False: product(q, tw, A[torch.from_numpy(need).to(DEV)].cpu().numpy(), Fs)}
    for flagged, p in enumerate(plans(q, tw)):
        for shared in (False, True):
            for count in counts[shared]:
                o = torch.full((count, k, N), -7, dtype=torch.int32, device=DEV)
                if shared:
                    p.matvec_shared(o, A_sh, s[:count], k, l)
                else:
                    p.matvec(o, A[:count], s[:count], k, l)
                torch.cuda.synchronize()
                idx = picks[(shared, count)]
                got = o[torch.from_numpy(idx).to(DEV)].cpu().numpy()
                assert_exact(got, exp[shared][pos[idx]], "q=%d k=%d l=%d %s, %s plan, count %d (grid-full %d) [%s]" % (
                    q, k, l, "matvec_shared" if shared else "matvec", plan_name(flagged), count,
                    G[shared], route(q, k, l, 0, flagged, shared)), index=idx)


@gpu_test
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG], ids=["chacha", "aes"])
@pytest.mark.parametrize("q,tw,k,l,q_bits,transposes", RAND_SHAPES)
def test_rand_products_exact(prng, q, tw, k, l, q_bits, transposes, arith, plans):
    """rand_product (one seed per instance), rand_product_shared (one seed) and both _host twins, fed the matrix
    rand_matrix draws, against the exact reference; y is any SINT32 on the default plan."""
    rng = np.random.default_rng(q + 10 * k + prng)
    A, snames, s, _ = exact_case(q, tw, k, l)
    for flagged, p in enumerate(plans(q, tw)):
        if l > lmax(q, arith):
            z = torch.zeros((3, l, N), dtype=torch.int32, device=DEV)
            refused(lambda: p.rand_product(torch.zeros((3, k, N), dtype=torch.int32, device=DEV), z,
                                           torch.zeros((3, 32), dtype=torch.uint8, device=DEV), prng, q_bits, k, l))
            refused(lambda: p.rand_product_shared(torch.zeros((3, k, N), dtype=torch.int32, device=DEV), z,
                                                  torch.zeros((32,), dtype=torch.uint8, device=DEV), prng, q_bits, k, l))
            continue
        sidx = [i for i, n in enumerate(snames) if n in S_IN or not flagged]
        y = np.concatenate([s[sidx], s[sidx]])                # each pattern under two seeds
        count = y.shape[0]
        names = ["y %s" % snames[i] for i in sidx] * 2
        seeds = rng.integers(0, 256, size=(count, 32)).astype(np.uint8)
        Fy = forward(q, tw, y)
        for transpose in transposes:
            label = "q=%d k=%d l=%d arith=%s %s plan transpose=%s" % (q, k, l, ARITH_IDS[arith], plan_name(flagged), transpose)
            M = torch.empty((count, k, l, N), dtype=torch.int32, device=DEV)
            B.rand_matrix(M, torch.from_numpy(seeds).to(DEV), prng, q, q_bits, N, k, l, transpose)
            torch.cuda.synchronize()
            exp = product(q, tw, M.cpu().numpy(), Fy)
            t = torch.full((count, k, N), -7, dtype=torch.int32, device=DEV)
            p.rand_product(t, dev(y), torch.from_numpy(seeds).to(DEV), prng, q_bits, k, l, transpose)
            torch.cuda.synchronize()
            assert_exact(t.cpu().numpy(), exp, label + " rand_product [%s]" % route(q, k, l, arith, flagged, False), names)
            th = np.full((count, k, N), -5, dtype=np.int32)
            p.rand_product_host(th, y, seeds, prng, q_bits, k, l, transpose)
            assert_exact(th, exp, label + " rand_product_host", names)
            exp_sh = product(q, tw, M[0].cpu().numpy(), Fy)
            t = torch.full((count, k, N), -7, dtype=torch.int32, device=DEV)
            p.rand_product_shared(t, dev(y), torch.from_numpy(seeds[0]).to(DEV), prng, q_bits, k, l, transpose)
            torch.cuda.synchronize()
            assert_exact(t.cpu().numpy(), exp_sh, label + " rand_product_shared [%s]" % route(q, k, l, arith, flagged, True),
                         names)
            th = np.full((count, k, N), -5, dtype=np.int32)
            p.rand_product_shared_host(th, y, np.ascontiguousarray(seeds[0]), prng, q_bits, k, l, transpose)
            assert_exact(th, exp_sh, label + " rand_product_shared_host", names)


@gpu_test
def test_refusals_under_every_arithmetic(arith, plans):
    """l = 6, 7, 8 on q = 8380417 (above sh32_mv_lmax = 5) and l = 5 on the small moduli are refused by every entry point
    under every arithmetic, on both plans; l = 5 on q = 8380417 is refused exactly where lmax() says so."""
    z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=DEV)  # noqa: E731
    seed = torch.zeros((32,), dtype=torch.uint8, device=DEV)
    cases = [(8380417, 32, 23, k, l) for l in (6, 7, 8) for k in (1, 6)] + \
            [(q, 16, qb, k, 5) for q, qb in ((7681, 13), (12289, 14)) for k in (1, 4)]
    if lmax(8380417, arith) < 5:
        cases.append((8380417, 32, 23, 6, 5))
    for q, tw, q_bits, k, l in cases:
        for p in plans(q, tw):
            c = 4
            refused(lambda: p.matvec(z(c, k, N), z(c, k, l, N), z(c, l, N), k, l))
            refused(lambda: p.matvec_shared(z(c, k, N), z(k, l, N), z(c, l, N), k, l))
            refused(lambda: p.rand_product(z(c, k, N), z(c, l, N), torch.zeros((c, 32), dtype=torch.uint8, device=DEV),
                                           sc.PRNG_CHACHA, q_bits, k, l))
            refused(lambda: p.rand_product_shared(z(c, k, N), z(c, l, N), seed, sc.PRNG_CHACHA, q_bits, k, l))
            refused(lambda: p.rand_product_host(np.zeros((c, k, N), np.int32), np.zeros((c, l, N), np.int32),
                                                np.zeros((c, 32), np.uint8), sc.PRNG_CHACHA, q_bits, k, l))
            refused(lambda: p.rand_product_shared_host(np.zeros((c, k, N), np.int32), np.zeros((c, l, N), np.int32),
                                                       np.zeros(32, np.uint8), sc.PRNG_CHACHA, q_bits, k, l))
