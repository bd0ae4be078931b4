"""The fused product n = 512, q = 12289 with the pass-0 entries of the reference's table compiled in as instruction
immediates (ntt_fast_fq32.cu: ArFqImm).  A plan whose derived entries equal the compiled ones runs that kernel; any
other table -- here the table of another primitive 2n-th root, which gives the same products -- runs the table-driven
kernel.  Both must give the oracle's bits on every input class the fused product accepts."""
import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import libsafecrypto_b200 as sc  # noqa: E402

Q, N = 12289, 512
DEV = "cuda:0"


def perturbed_tables():
    """The reference's layout (w[i] = g^i, r[i] = -(n^-1) g^i) for g = psi^3, another primitive 2n-th root."""
    w, _ = O.tables(Q, N, 16)
    g = pow(int(w[1]), 3, Q)
    ninv = pow(N, Q - 2, Q)
    wp = [pow(g, i, Q) for i in range(N)]
    rp = [(Q - ninv) * x % Q for x in wp]
    assert pow(g, N, Q) == Q - 1 and wp != [int(x) for x in w]
    return np.array(wp, dtype=np.int16), np.array(rp, dtype=np.int16)


_plans = {}


def plan(kind, in_range):
    key = (kind, in_range)
    if key not in _plans:
        w, r = O.tables(Q, N, 16) if kind == "reference" else perturbed_tables()
        p = sc.NttPlan(N, Q, sc.REFERENCE, w, r)
        if in_range:
            p.set_flags(sc.PLAN_INPUTS_IN_RANGE)
        _plans[key] = p
    return _plans[key]


def kernels_of(fn):
    """Names of the fused-product kernels fn launches."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if "k_polymul_w32" in e.name}


def expected(a, b):
    w, r = O.tables(Q, N, 16)
    return O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, N, Q, 16, np.mod(a, Q).astype(np.int32),
                              np.mod(b, Q).astype(np.int32), w, r)


@pytest.mark.parametrize("in_range", [True, False])
def test_compiled_table_is_chosen_only_for_the_reference_table(in_range):
    rng = np.random.default_rng(11)
    a = torch.from_numpy(rng.integers(0, Q, size=(64, N)).astype(np.int32)).to(DEV)
    b = torch.from_numpy(rng.integers(0, Q, size=(64, N)).astype(np.int32)).to(DEV)
    out = torch.empty_like(a)
    ref = kernels_of(lambda: plan("reference", in_range).polymul(out, a, b))
    per = kernels_of(lambda: plan("perturbed", in_range).polymul(out, a, b))
    assert ref and all("ArFqImm" in k for k in ref), ref
    assert per and not any("ArFqImm" in k for k in per), per


def inputs(rng, kind, rows):
    if kind == "uniform":
        return rng.integers(0, Q, size=(rows, N)), rng.integers(0, Q, size=(rows, N))
    if kind == "edge":                                  # |x| = 4q, the bound of the in-range plan, adversarial signs
        s = rng.choice([-1, 1], size=(2, rows, N))
        a, b = 4 * Q * s[0], 4 * Q * s[1]
        a[:, ::3] = 4 * Q
        b[:, 1::3] = -4 * Q
        return a, b
    if kind == "signed":
        return rng.integers(-4 * Q, 4 * Q + 1, size=(rows, N)), rng.integers(-4 * Q, 4 * Q + 1, size=(rows, N))
    x = rng.integers(-2**31, 2**31, size=(2, rows, N))     # full SINT32 range: the checked plan only
    x[0, 0, :4] = [2**31 - 1, -2**31, -1, 4 * Q + 1]
    return x[0], x[1]


@pytest.mark.parametrize("table", ["reference", "perturbed"])
@pytest.mark.parametrize("in_range", [True, False])
@pytest.mark.parametrize("kind", ["uniform", "edge", "signed", "sint32"])
def test_products_match_the_oracle(table, in_range, kind):
    if in_range and kind == "sint32":
        pytest.skip("the in-range plan takes |x| <= 4q")
    rng = np.random.default_rng([len(table), int(in_range), len(kind)])
    p = plan(table, in_range)
    for rows in (1, 7, 33, 161, 20000):                 # ragged counts, and batches beyond one grid (work counter)
        a, b = (x.astype(np.int32) for x in inputs(rng, kind, rows))
        exp = expected(a, b)
        out = torch.full((rows, N), -7, dtype=torch.int32, device=DEV)
        p.polymul(out, torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV))
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), exp), (rows,)


@pytest.mark.parametrize("table", ["reference", "perturbed"])
@pytest.mark.parametrize("in_range", [True, False])
def test_unaligned_rows(table, in_range):
    """Rows that are not 16-byte aligned take the plain-load (LDG) variant of the kernel."""
    rng = np.random.default_rng(5)
    p = plan(table, in_range)
    for rows in (1, 33, 161):
        a, b = (x.astype(np.int32) for x in inputs(rng, "signed", rows))
        exp = expected(a, b)
        for off_a, off_b in ((1, 0), (0, 3), (2, 1)):
            da = torch.zeros(rows * N + 8, dtype=torch.int32, device=DEV)
            db = torch.zeros(rows * N + 8, dtype=torch.int32, device=DEV)
            da[off_a:off_a + rows * N] = torch.from_numpy(a).to(DEV).reshape(-1)
            db[off_b:off_b + rows * N] = torch.from_numpy(b).to(DEV).reshape(-1)
            out = torch.full((rows, N), -7, dtype=torch.int32, device=DEV)
            p.polymul(out, da[off_a:off_a + rows * N].view(rows, N), db[off_b:off_b + rows * N].view(rows, N))
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), exp), (rows, off_a, off_b)
