"""Products with the error term added in the same call (scgpu_polymul_add_batch, scgpu_ntt_mul_key_add_batch,
scgpu_matvec_add_batch, scgpu_matvec_shared_add_batch): bit for bit (P + e) mod q, P the sibling call's result, under
every arithmetic and on both plans; checked against the sibling, against a schoolbook product in Python integers, for
addends at the edges of their range, in place, on unaligned rows, over batch sizes around the grid and the claim phases,
for the sibling's refusals, and for one launch per call (the epilogue of the warp-local kernels)."""
import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import libsafecrypto_b200 as sc  # noqa: E402

DEV = "cuda:0"
ERR_ARG, ERR_UNSUPPORTED = -1, -3
I32_MIN, I32_MAX = -2**31, 2**31 - 1

# (q, n, table): "ref" = the reference's table (n = 512, q = 12289: the compiled-immediate kernel), "psi3" = the
# reference's layout for psi^3 (the table-driven kernel of the same shape)
RINGS = [(12289, 512, "ref"), (12289, 512, "psi3"), (12289, 1024, "ref"), (7681, 256, "ref"), (18433, 512, "ref"),
         (8380417, 256, "ref"), (51750913, 512, "ref")]
MODULES = [(7681, 2, 2), (7681, 3, 3), (7681, 4, 4), (7681, 3, 2),
           (8380417, 5, 4), (8380417, 6, 5), (8380417, 3, 2), (8380417, 1, 5)]


def tw_bits(q):
    return 16 if q < 32768 else 32


def tables(q, n, kind):
    w, r = O.tables(q, n, tw_bits(q))
    if kind == "ref":
        return w, r
    g = pow(int(w[1]), 3, q)
    ninv = pow(n, q - 2, q)
    wp = [pow(g, i, q) for i in range(n)]
    rp = [(q - ninv) * x % q for x in wp]
    assert pow(g, n, q) == q - 1
    dt = np.int16 if tw_bits(q) == 16 else np.int32
    return np.array(wp, dtype=dt), np.array(rp, dtype=dt)


_plans = {}


def plan(q, n, kind="ref", in_range=False):
    key = (q, n, kind, in_range)
    if key not in _plans:
        w, r = tables(q, n, kind)
        p = sc.NttPlan(n, q, sc.REFERENCE, w, r)
        if in_range:
            p.set_flags(sc.PLAN_INPUTS_IN_RANGE)
        _plans[key] = p
    return _plans[key]


@pytest.fixture(params=["auto", "montgomery", "barrett32", "fq8", "shoup", "force_montgomery"])
def arith(request):
    """Every arithmetic of scgpu_set_fast_arith, and scgpu_force_montgomery."""
    L = sc.lib()
    modes = {"auto": 0, "montgomery": 1, "barrett32": 2, "fq8": 3, "shoup": 4}
    if request.param == "force_montgomery":
        old = L.scgpu_set_fast_arith(0)
        L.scgpu_force_montgomery(1)
    else:
        old = L.scgpu_set_fast_arith(modes[request.param])
    yield request.param
    L.scgpu_set_fast_arith(old)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def operands(rng, q, shape, in_range):
    """Canonical, centred and (default plan) full-range SINT32 coefficients, mixed."""
    x = rng.integers(0, q, size=shape, dtype=np.int64)
    sel = rng.integers(0, 4, size=shape)
    x = np.where(sel == 1, rng.integers(-4 * q, 4 * q + 1, size=shape), x)
    if not in_range:
        x = np.where(sel == 2, rng.integers(I32_MIN, I32_MAX + 1, size=shape, dtype=np.int64), x)
    return x.astype(np.int32)


def addend(rng, q, shape, in_range):
    """Small errors, the +-4q edges and (default plan) the whole SINT32 range with its two ends."""
    e = rng.integers(-8, 9, size=shape, dtype=np.int64)
    sel = rng.integers(0, 5, size=shape)
    e = np.where(sel == 1, rng.choice(np.array([-4 * q, 4 * q, -4 * q + 1, 4 * q - 1]), size=shape), e)
    e = np.where(sel == 2, rng.integers(-4 * q, 4 * q + 1, size=shape), e)
    if not in_range:
        e = np.where(sel == 3, rng.integers(I32_MIN, I32_MAX + 1, size=shape, dtype=np.int64), e)
        e = np.where(sel == 4, rng.choice(np.array([I32_MIN, I32_MAX, I32_MIN + 1, I32_MAX - 1]), size=shape), e)
    return e.astype(np.int32)


def plus(P, e, q):
    return np.mod(P.cpu().numpy().astype(np.int64) + e.cpu().numpy().astype(np.int64), q).astype(np.int32)


# ---- 1. composition: every shape, arithmetic and plan -----------------------------------------------------------------

@pytest.mark.parametrize("in_range", [False, True], ids=["default", "in_range"])
@pytest.mark.parametrize("q,n,kind", RINGS)
def test_polymul_add_is_sibling_plus_e(q, n, kind, in_range, arith):
    rng = np.random.default_rng(q + n + in_range)
    p = plan(q, n, kind, in_range)
    count = 301
    a, b = dev(operands(rng, q, (count, n), in_range)), dev(operands(rng, q, (count, n), in_range))
    e = dev(addend(rng, q, (count, n), in_range))
    P = torch.empty_like(a)
    for bb in (b, b[7].contiguous()):                             # per-row and one shared second operand (b_stride = 0)
        p.polymul(P, a, bb)
        out = torch.full_like(a, -5)
        p.polymul_add(out, a, bb, e)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), plus(P, e, q))


@pytest.mark.parametrize("in_range", [False, True], ids=["default", "in_range"])
@pytest.mark.parametrize("q,n,kind", [r for r in RINGS if r[2] == "ref"])
def test_mul_key_add_is_sibling_plus_e(q, n, kind, in_range, arith):
    rng = np.random.default_rng(q + 3 * n + in_range)
    p = plan(q, n, kind, in_range)
    count = 263
    t = dev(operands(rng, q, (count, n), in_range))
    e = dev(addend(rng, q, (count, n), in_range))
    widths = [torch.int32] + ([torch.int16] if q < 32768 else [])
    for dt in widths:
        keys = dev(rng.integers(0, q, size=(count, n)).astype(np.int64)).to(dt)
        for key in (keys, keys[3].contiguous()):                  # per row, and key_stride = 0 (the residue-table route)
            P = torch.empty_like(t)
            p.mul_key(P, t, key)
            out = torch.full_like(t, -5)
            p.mul_key_add(out, t, key, e)
            torch.cuda.synchronize()
            assert np.array_equal(out.cpu().numpy(), plus(P, e, q)), (dt, key.dim())


@pytest.mark.parametrize("one_warp", [False, True], ids=["default_kernels", "one_warp"])
@pytest.mark.parametrize("in_range", [False, True], ids=["default", "in_range"])
@pytest.mark.parametrize("q,k,l", MODULES)
def test_matvec_add_is_sibling_plus_e(q, k, l, in_range, one_warp, arith, monkeypatch):
    if one_warp:
        monkeypatch.setenv("SCGPU_MATVEC_ONE_WARP", "1")
    rng = np.random.default_rng(q + 10 * k + l + in_range)
    p = plan(q, 256, "ref", in_range)
    count = 197
    A = dev(operands(rng, q, (count, k, l, 256), in_range))
    s = dev(operands(rng, q, (count, l, 256), in_range))
    e = dev(addend(rng, q, (count, k, 256), in_range))
    P = torch.empty((count, k, 256), dtype=torch.int32, device=DEV)
    try:
        p.matvec(P, A, s, k, l)
    except sc.ScgpuError as refused:
        # the sibling refuses this (k, l) under this arithmetic: so must the add call, with the same status
        with pytest.raises(sc.ScgpuError) as also:
            p.matvec_add(P, A, s, e, k, l)
        assert str(refused).rsplit("(status", 1)[1] == str(also.value).rsplit("(status", 1)[1]
        return
    out = torch.full_like(P, -5)
    p.matvec_add(out, A, s, e, k, l)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), plus(P, e, q))
    A0 = A[5].contiguous()
    p.matvec_shared(P, A0, s, k, l)
    out.fill_(-5)
    p.matvec_shared_add(out, A0, s, e, k, l)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), plus(P, e, q))


# ---- 2. independent check: schoolbook negacyclic products in Python integers -------------------------------------------

def negacyclic(a, b, q):
    a = [int(x) % q for x in a]
    b = [int(x) % q for x in b]
    n = len(a)
    c = [0] * n
    for i, x in enumerate(a):
        if x == 0:
            continue
        for j, y in enumerate(b):
            k = i + j
            if k < n:
                c[k] += x * y
            else:
                c[k - n] -= x * y
    return c


@pytest.mark.parametrize("in_range", [False, True], ids=["default", "in_range"])
@pytest.mark.parametrize("q,n", [(12289, 512), (12289, 1024), (7681, 256), (18433, 512), (8380417, 256), (51750913, 512)])
def test_schoolbook_rows(q, n, in_range):
    rng = np.random.default_rng(q ^ n)
    p = plan(q, n, "ref", in_range)
    count = 65
    a, b = operands(rng, q, (count, n), in_range), operands(rng, q, (count, n), in_range)
    e = addend(rng, q, (count, n), in_range)
    out = torch.empty((count, n), dtype=torch.int32, device=DEV)
    p.polymul_add(out, dev(a), dev(b), dev(e))
    # the key product: the key is the forward transform of a time-domain polynomial kt (the reference's NTT-domain order)
    kt = rng.integers(0, q, size=(count, n)).astype(np.int32)
    key = torch.empty_like(out)
    p.ntt_canonical(key, dev(kt))
    ok = torch.empty_like(out)
    p.mul_key_add(ok, dev(a), key, dev(e))
    torch.cuda.synchronize()
    got, gotk = out.cpu().numpy(), ok.cpu().numpy()
    for row in (0, 31, count - 1):
        want = [(c + int(x)) % q for c, x in zip(negacyclic(a[row], b[row], q), e[row])]
        assert [int(v) for v in got[row]] == want, row
        want = [(c + int(x)) % q for c, x in zip(negacyclic(a[row], kt[row], q), e[row])]
        assert [int(v) for v in gotk[row]] == want, row


@pytest.mark.parametrize("q,k,l", [(7681, 3, 3), (8380417, 5, 4)])
def test_schoolbook_module_rows(q, k, l):
    rng = np.random.default_rng(q + k)
    p = plan(q, 256, "ref", False)
    count = 9
    at = rng.integers(0, q, size=(count, k, l, 256)).astype(np.int32)
    A = torch.empty((count * k * l, 256), dtype=torch.int32, device=DEV)
    p.ntt_canonical(A, dev(at.reshape(-1, 256)))
    A = A.view(count, k, l, 256)
    s = operands(rng, q, (count, l, 256), False)
    e = addend(rng, q, (count, k, 256), False)
    out = torch.empty((count, k, 256), dtype=torch.int32, device=DEV)
    p.matvec_add(out, A, dev(s), dev(e), k, l)
    sh = torch.empty_like(out)
    p.matvec_shared_add(sh, A[2].contiguous(), dev(s), dev(e), k, l)
    torch.cuda.synchronize()
    got, gots = out.cpu().numpy(), sh.cpu().numpy()
    for inst in (0, count - 1):
        for i in range(k):
            acc = [0] * 256
            accs = [0] * 256
            for j in range(l):
                acc = [x + y for x, y in zip(acc, negacyclic(at[inst, i, j], s[inst, j], q))]
                accs = [x + y for x, y in zip(accs, negacyclic(at[2, i, j], s[inst, j], q))]
            assert [int(v) for v in got[inst, i]] == [(c + int(x)) % q for c, x in zip(acc, e[inst, i])]
            assert [int(v) for v in gots[inst, i]] == [(c + int(x)) % q for c, x in zip(accs, e[inst, i])]


# ---- 3. addend patterns ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("in_range", [False, True], ids=["default", "in_range"])
@pytest.mark.parametrize("q,n", [(12289, 512), (8380417, 256), (51750913, 512)])
def test_addend_patterns(q, n, in_range):
    rng = np.random.default_rng(7 * q + n)
    p = plan(q, n, "ref", in_range)
    count = 130
    a, b = dev(operands(rng, q, (count, n), in_range)), dev(operands(rng, q, (count, n), in_range))
    P = torch.empty_like(a)
    p.polymul(P, a, b)
    pats = {"zero": np.zeros((count, n), np.int64),
            "edges": rng.choice(np.array([-4 * q, 4 * q]), size=(count, n)),
            "small": rng.integers(-3, 4, size=(count, n))}
    if not in_range:
        pats["full"] = rng.integers(I32_MIN, I32_MAX + 1, size=(count, n), dtype=np.int64)
        pats["ends"] = rng.choice(np.array([I32_MIN, I32_MAX]), size=(count, n))
    for name, ev in pats.items():
        e = dev(ev.astype(np.int32))
        out = torch.full_like(a, -5)
        p.polymul_add(out, a, b, e)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), plus(P, e, q)), name
        if name == "zero":
            assert torch.equal(out, P)


# ---- 4. aliasing and alignment -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("q,n", [(12289, 512), (8380417, 256)])
def test_in_place_and_unaligned(q, n, arith):
    rng = np.random.default_rng(q + 99)
    p = plan(q, n)
    count = 77
    a, b = dev(operands(rng, q, (count, n), False)), dev(operands(rng, q, (count, n), False))
    e = dev(addend(rng, q, (count, n), False))
    P = torch.empty_like(a)
    p.polymul(P, a, b)
    want = plus(P, e, q)
    acc = e.clone()
    p.polymul_add(acc, a, b, acc)                               # out is e: out += a b
    torch.cuda.synchronize()
    assert np.array_equal(acc.cpu().numpy(), want)

    def shifted(x):                                           # rows 4 bytes off a 16-byte boundary
        buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=DEV)
        v = buf[1:].view(x.shape)
        v.copy_(x)
        return v
    ua, ub, ue, uo = shifted(a), shifted(b), shifted(e), shifted(torch.zeros_like(a))
    p.polymul_add(uo, ua, ub, ue)
    torch.cuda.synchronize()
    assert np.array_equal(uo.cpu().numpy(), want)
    p.polymul_add(ue, ua, ub, ue)                               # in place on unaligned rows
    torch.cuda.synchronize()
    assert np.array_equal(ue.cpu().numpy(), want)
    if n == 256:
        k, l = (3, 2) if q < 59000 else (5, 4)
        A = dev(rng.integers(0, q, size=(count, k, l, n)).astype(np.int32))
        s = dev(operands(rng, q, (count, l, n), False))
        em = dev(addend(rng, q, (count, k, n), False))
        M = torch.empty((count, k, n), dtype=torch.int32, device=DEV)
        p.matvec(M, A, s, k, l)
        want = plus(M, em, q)
        acc = em.clone()
        p.matvec_add(acc, A, s, acc, k, l)
        mo = shifted(torch.zeros_like(M))
        p.matvec_add(mo, shifted(A), shifted(s), shifted(em), k, l)
        torch.cuda.synchronize()
        assert np.array_equal(acc.cpu().numpy(), want)
        assert np.array_equal(mo.cpu().numpy(), want)


# ---- 5. batch sizes ----------------------------------------------------------------------------------------------------

def test_batch_sizes_around_the_grid_and_the_claim_phases():
    q, n = 12289, 512
    p = plan(q, n)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid = sms * 20 * 2                                       # products in one grid-full of k_polymul_w32 (n = 512)
    biggest = 12 * grid + 3                                   # chunked claims run up to 10 grid-fulls before the end
    g = torch.Generator(device=DEV).manual_seed(5)
    a = torch.randint(0, q, (biggest, n), dtype=torch.int32, device=DEV, generator=g)
    b = torch.randint(0, q, (biggest, n), dtype=torch.int32, device=DEV, generator=g)
    e = torch.randint(-4 * q, 4 * q + 1, (biggest, n), dtype=torch.int32, device=DEV, generator=g)
    P = torch.empty_like(a)
    p.polymul(P, a, b)
    want = torch.remainder(P.long() + e.long(), q).int()
    for count in (0, 1, 2, 3, 333, grid - 1, grid, grid + 1, 2 * grid + 1, 10 * grid - 1, 10 * grid, 10 * grid + 1, biggest):
        out = torch.full_like(a, -5)
        p.polymul_add(out, a, b, e, count=count)
        torch.cuda.synchronize()
        assert torch.equal(out[:count], want[:count]), count
        assert bool((out[count:] == -5).all()), count
    for k, l, qq in ((3, 3, 7681), (5, 4, 8380417)):
        pm = plan(qq, 256)
        cnt = 3 * sms * 16 * 4 + 5
        A = torch.randint(0, qq, (k, l, 256), dtype=torch.int32, device=DEV, generator=g)
        s = torch.randint(-5, 6, (cnt, l, 256), dtype=torch.int32, device=DEV, generator=g)
        em = torch.randint(-9, 10, (cnt, k, 256), dtype=torch.int32, device=DEV, generator=g)
        M = torch.empty((cnt, k, 256), dtype=torch.int32, device=DEV)
        pm.matvec_shared(M, A, s, k, l)
        want = torch.remainder(M.long() + em.long(), qq).int()
        for count in (0, 1, 5, cnt):
            out = torch.full_like(M, -5)
            pm.matvec_shared_add(out, A, s, em, k, l, count=count)
            torch.cuda.synchronize()
            assert torch.equal(out[:count], want[:count]), (k, l, count)
            assert bool((out[count:] == -5).all())


# ---- 6. refusals -------------------------------------------------------------------------------------------------------

def test_refusals_follow_the_sibling():
    L = sc.lib()
    st = torch.cuda.current_stream().cuda_stream
    p = plan(7681, 256)
    x = torch.zeros((4, 4, 9, 256), dtype=torch.int32, device=DEV)
    e = torch.zeros((4, 9, 256), dtype=torch.int32, device=DEV)
    P = sc.binding._ptr
    h = p.handle
    assert L.scgpu_polymul_add_batch(h, P(e), P(x), P(x), 256, None, 4, st) == ERR_ARG
    assert L.scgpu_ntt_mul_key_add_batch(h, P(e), P(x), P(x), 32, 256, None, 4, st) == ERR_ARG
    assert L.scgpu_matvec_add_batch(h, P(e), P(x), P(x), None, 2, 2, 4, st) == ERR_ARG
    assert L.scgpu_matvec_shared_add_batch(h, P(e), P(x), P(x), None, 2, 2, 4, st) == ERR_ARG
    assert L.scgpu_polymul_add_batch(None, P(e), P(x), P(x), 256, P(e), 4, st) == ERR_ARG
    for k, l in ((2, 9), (0, 2), (2, 0), (3, 5)):               # l beyond lmax of the modulus, empty shapes
        for sib, add in ((L.scgpu_matvec_batch, L.scgpu_matvec_add_batch),
                         (L.scgpu_matvec_shared_batch, L.scgpu_matvec_shared_add_batch)):
            want = sib(h, P(e), P(x), P(x), k, l, 4, st)
            assert want < 0
            assert add(h, P(e), P(x), P(x), P(e), k, l, 4, st) == want, (k, l)
    for bits in (8, 64):
        want = L.scgpu_ntt_mul_key_batch(h, P(e), P(x), P(x), bits, 256, 4, st)
        assert want == ERR_ARG
        assert L.scgpu_ntt_mul_key_add_batch(h, P(e), P(x), P(x), bits, 256, P(e), 4, st) == want
    p512 = plan(12289, 512)                                   # the module products are instantiated for n = 256 only
    want = L.scgpu_matvec_batch(p512.handle, P(e), P(x), P(x), 2, 2, 4, st)
    assert want == ERR_UNSUPPORTED
    assert L.scgpu_matvec_add_batch(p512.handle, P(e), P(x), P(x), P(e), 2, 2, 4, st) == want
    assert L.scgpu_polymul_add_batch(h, P(e), P(x), P(x), 256, P(e), 0, st) == 0     # count = 0: nothing to do


# ---- 7. one launch -----------------------------------------------------------------------------------------------------

def kernel_names(fn):
    """Names of the library kernels the profiler saw fn() launch.  The profiler can lose kernel records (the launch
    counter above is what shows one launch per call), so fn is profiled again, up to three times, until a record shows."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = {ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA and "k_" in ev.name}
        if names:
            return names
    return set()


def test_one_launch_under_the_automatic_arithmetic():
    old = sc.lib().scgpu_set_fast_arith(0)
    try:
        g = torch.Generator(device=DEV).manual_seed(6)
        for q, n in ((12289, 512), (12289, 1024), (8380417, 256), (51750913, 512)):
            p = plan(q, n)
            a = torch.randint(0, q, (999, n), dtype=torch.int32, device=DEV, generator=g)
            e = torch.randint(-5, 6, (999, n), dtype=torch.int32, device=DEV, generator=g)
            out = torch.empty_like(a)
            for sib, add in ((lambda: p.polymul(out, a, a), lambda: p.polymul_add(out, a, a, e)),
                             (lambda: p.mul_key(out, a, a[0]), lambda: p.mul_key_add(out, a, a[0], e))):
                c0 = sc.launch_count(); sib(); c1 = sc.launch_count(); add(); c2 = sc.launch_count()
                assert c2 - c1 == c1 - c0, (q, n)
        for q, k, l in ((7681, 3, 3), (8380417, 5, 4)):
            p = plan(q, 256)
            A = torch.randint(0, q, (999, k, l, 256), dtype=torch.int32, device=DEV, generator=g)
            s = torch.randint(-5, 6, (999, l, 256), dtype=torch.int32, device=DEV, generator=g)
            e = torch.randint(-5, 6, (999, k, 256), dtype=torch.int32, device=DEV, generator=g)
            out = torch.empty_like(e)
            for sib, add in ((lambda: p.matvec(out, A, s, k, l), lambda: p.matvec_add(out, A, s, e, k, l)),
                             (lambda: p.matvec_shared(out, A[0], s, k, l), lambda: p.matvec_shared_add(out, A[0], s, e, k, l))):
                c0 = sc.launch_count(); sib(); c1 = sc.launch_count(); add(); c2 = sc.launch_count()
                assert c2 - c1 == c1 - c0, (q, k, l)
        # the headline shape runs the compiled-immediate product kernel, addend included
        p = plan(12289, 512)
        a = torch.randint(0, 12289, (999, 512), dtype=torch.int32, device=DEV, generator=g)
        e = torch.randint(-5, 6, (999, 512), dtype=torch.int32, device=DEV, generator=g)
        out = torch.empty_like(a)
        names = kernel_names(lambda: p.polymul_add(out, a, a, e))
        assert names and all("k_polymul_w32" in x and "ArFqImm" in x for x in names), names
        names = kernel_names(lambda: plan(12289, 512, "psi3").polymul_add(out, a, a, e))
        assert names and all("k_polymul_w32" in x and "ArFqImm" not in x for x in names), names
    finally:
        sc.lib().scgpu_set_fast_arith(old)


@pytest.mark.parametrize("q,k,l", [(7681, 3, 3), (8380417, 5, 4)])
def test_shared_add_in_a_cuda_graph(q, k, l):
    p = plan(q, 256)
    g = torch.Generator(device=DEV).manual_seed(8)
    count = 1 << 14
    A = torch.randint(0, q, (k, l, 256), dtype=torch.int32, device=DEV, generator=g)
    s = torch.randint(-5, 6, (count, l, 256), dtype=torch.int32, device=DEV, generator=g)
    e = torch.randint(-5, 6, (count, k, 256), dtype=torch.int32, device=DEV, generator=g)
    eager = torch.empty((count, k, 256), dtype=torch.int32, device=DEV)
    p.matvec_shared_add(eager, A, s, e, k, l)
    torch.cuda.synchronize()
    out = torch.zeros_like(eager)
    graph = torch.cuda.CUDAGraph()
    st = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(st):
        with torch.cuda.graph(graph, stream=st):
            p.matvec_shared_add(out, A, s, e, k, l, stream=st)
    for _ in range(2):
        out.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
