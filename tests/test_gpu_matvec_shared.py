"""Module products with ONE matrix for the whole batch (scgpu_matvec_shared_batch, scgpu_rand_product_csprng_shared_batch):
bit for bit the per-instance entry points with the matrix (or the seed) repeated for every instance, which the other
suites pin to the port, the compiled reference and tests/golden/golden_v3.npz.  Also checked here against the port
directly, and for refusals, concurrent streams on one plan and CUDA-graph capture."""
import os

import numpy as np
import pytest

import _oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import libsafecrypto_b200 as sc  # noqa: E402

DEV = "cuda:0"
N = 256
G3 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v3.npz")
KYBER = [(7681, 16, 2, 2), (7681, 16, 3, 3), (7681, 16, 4, 4), (7681, 16, 3, 2), (7681, 16, 2, 3), (12289, 16, 2, 2)]
DILITHIUM = [(8380417, 32, 5, 4), (8380417, 32, 6, 5), (8380417, 32, 3, 2), (8380417, 32, 8, 1), (8380417, 32, 1, 5)]
SHAPES = KYBER + DILITHIUM


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


@pytest.fixture(params=[0, 1, 2, 3, 4], ids=["auto", "montgomery", "barrett32", "fq8", "shoup"])
def arith(request):
    """Every arithmetic of scgpu_set_fast_arith: the shared path must follow the per-instance one in each."""
    old = sc.lib().scgpu_set_fast_arith(request.param)
    yield request.param
    sc.lib().scgpu_set_fast_arith(old)


def matrices(rng, q, k, l, in_range):
    """A uniform in [0, q), and one at the edges of the +-4q window (default plan: any SINT32 as well)."""
    x0 = 4 * q
    edge = rng.choice(np.array([-x0, x0, 0, q - 1], dtype=np.int64), size=(k, l, N)).astype(np.int32)
    out = [rng.integers(0, q, size=(k, l, N)).astype(np.int32), edge]
    if not in_range:
        out.append(rng.integers(-2**31, 2**31, size=(k, l, N), dtype=np.int64).astype(np.int32))
    return out


def shared_and_replicated(p, A, s, k, l, count):
    """(matvec_shared, matvec with A expanded to count copies) on device tensors."""
    o1 = torch.full((count, k, N), -7, dtype=torch.int32, device=DEV)
    o2 = torch.full((count, k, N), -9, dtype=torch.int32, device=DEV)
    p.matvec_shared(o1, A, s, k, l, count=count)
    p.matvec(o2, A.unsqueeze(0).expand(count, k, l, N).contiguous(), s, k, l, count=count)
    torch.cuda.synchronize()
    return o1, o2


def grid_instances(q, k, l):
    """Instances in one grid-full of the shared kernel launch_matvec_w32 picks under the automatic arithmetic."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if q < 59000:                                              # k_matvec16_w32: 4 instances per one-warp CTA
        smem = (4 * (296 + 264) + l * 4 * 168) * 4
        return sms * min(16, (227 * 1024) // (smem + 1088)) * 4
    if 2 <= k <= 8:                                            # k_matvec_rows_w32: 4 instances per CTA of k warps
        smem = (l + k) * 4 * 296 * 4
        return sms * max(1, min((227 * 1024) // (smem + 1280), 65536 // (k * 32 * 128))) * 4
    smem = ((l + 1) * 4 * 296 + 4 * 264) * 4                   # k_matvec_w32
    return sms * min(16, (227 * 1024) // (smem + 1088)) * 4


@pytest.mark.parametrize("q,tw,k,l", SHAPES)
def test_shared_equals_replicated(q, tw, k, l, arith, plans):
    """Small batches, every arithmetic, default and in-range plans, matrices in [0, q) and at the window edges."""
    if l > 4 and arith in (1, 2, 3):
        pytest.skip("l > 4 is only instantiated for the Shoup-policy kernels")
    rng = np.random.default_rng(1000 * k + 10 * l + arith)
    for flagged, p in enumerate(plans(q, tw)):
        for A in matrices(rng, q, k, l, flagged):
            for count in (1, 3, 37):
                s = rng.integers(-4 * q, 4 * q + 1, size=(count, l, N)).astype(np.int32)
                s[count // 2:] = rng.integers(-5, 6, size=(count - count // 2, l, N))
                o1, o2 = shared_and_replicated(p, torch.from_numpy(A).to(DEV), torch.from_numpy(s).to(DEV), k, l, count)
                assert torch.equal(o1, o2), (flagged, count)
                assert int(o1.min()) >= 0 and int(o1.max()) < q


@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (7681, 16, 2, 2), (8380417, 32, 5, 4), (8380417, 32, 6, 5),
                                      (8380417, 32, 1, 5)])
def test_shared_equals_replicated_across_grid_fulls(q, tw, k, l, plans):
    """One grid-full -1 / +0 / +1 and twelve grid-fulls plus a ragged tail: the work counter's chunked and single-group
    phases both run."""
    g = torch.Generator(device=DEV).manual_seed(q + k + l)
    G = grid_instances(q, k, l)
    for p in plans(q, tw):
        A = torch.randint(0, q, (k, l, N), dtype=torch.int32, device=DEV, generator=g)
        for count in (G - 1, G, G + 1, 12 * G + 5):
            s = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
            o1, o2 = shared_and_replicated(p, A, s, k, l, count)
            assert torch.equal(o1, o2), count


@pytest.mark.parametrize("var", ["SCGPU_MATVEC_ONE_WARP", "SCGPU_MATVEC_STASH32", "SCGPU_MATVEC_FLOAT_ACC"])
@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (7681, 16, 4, 4), (8380417, 32, 5, 4), (8380417, 32, 6, 5)])
def test_kernel_selection_variables(var, q, tw, k, l, plans, monkeypatch):
    """The launch-time variables pick other kernels for both entry points alike."""
    monkeypatch.setenv(var, "1")
    g = torch.Generator(device=DEV).manual_seed(7)
    G = grid_instances(q, k, l)
    for p in plans(q, tw):
        A = torch.randint(0, q, (k, l, N), dtype=torch.int32, device=DEV, generator=g)
        for count in (37, 3 * G + 1):
            s = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
            o1, o2 = shared_and_replicated(p, A, s, k, l, count)
            assert torch.equal(o1, o2), count


@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (7681, 16, 2, 3), (8380417, 32, 5, 4), (8380417, 32, 1, 5)])
def test_unaligned_rows(q, tw, k, l, plans):
    """s and out one word off a 16-byte boundary: the plain-load kernels (no bulk copies of s)."""
    rng = np.random.default_rng(q + 3)
    count = 300
    for p in plans(q, tw):
        A = torch.from_numpy(rng.integers(0, q, size=(k, l, N)).astype(np.int32)).to(DEV)
        sb = torch.from_numpy(rng.integers(-5, 6, size=(count * l * N + 1,)).astype(np.int32)).to(DEV)
        s = sb[1:].view(count, l, N)
        ob = torch.full((count * k * N + 1,), -7, dtype=torch.int32, device=DEV)
        o1 = ob[1:].view(count, k, N)
        o2 = torch.empty((count, k, N), dtype=torch.int32, device=DEV)
        p.matvec_shared(o1, A, s, k, l)
        p.matvec(o2, A.unsqueeze(0).expand(count, k, l, N).contiguous(), s, k, l)
        torch.cuda.synchronize()
        assert torch.equal(o1, o2)
        # the unaligned matrix itself (the stride-0 kernels read it in place)
        Ab = torch.empty((k * l * N + 1,), dtype=torch.int32, device=DEV)
        Ab[1:] = A.reshape(-1)
        o3 = torch.empty_like(o2)
        p.matvec_shared(o3, Ab[1:].view(k, l, N), s, k, l)
        torch.cuda.synchronize()
        assert torch.equal(o3, o2)


@pytest.mark.parametrize("q,tw,k,l,eta", [(7681, 16, 3, 3, 4), (7681, 16, 2, 3, 5), (8380417, 32, 6, 5, 5), (8380417, 32, 8, 1, 2)])
def test_against_the_port(q, tw, k, l, eta, arith, plans):
    """t_i = normalize(inv_ntt(normalize(sum_j A_ij o fwd_ntt(s_j)))) through the port, independently of the kernels."""
    if l > 4 and arith in (1, 2, 3):
        pytest.skip("l > 4 is only instantiated for the Shoup-policy kernels")
    count = 41
    rng = np.random.default_rng(q + 10 * k + l)
    w, r = O.tables(q, N, tw)
    A = rng.integers(0, q, size=(k, l, N)).astype(np.int32)
    s = rng.integers(-eta, eta + 1, size=(count, l, N)).astype(np.int32)
    P = O.port()
    sh = P.ntt_batch(O.REFERENCE, O.OP_FWD, N, q, tw, s.reshape(-1, N), None, w, r).reshape(count, l, N)
    exp = np.zeros((count, k, N), dtype=np.int32)
    for i in range(k):
        acc = np.zeros((count, N), dtype=np.int64)
        for j in range(l):
            acc += P.ntt_batch(O.REFERENCE, O.OP_PW, N, q, tw, np.tile(A[i, j], (count, 1)), sh[:, j])
        t = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, N, q, tw, acc.astype(np.int32))
        t = P.ntt_batch(O.REFERENCE, O.OP_INV, N, q, tw, t, None, w, r)
        exp[:, i] = P.ntt_batch(O.REFERENCE, O.OP_NORMALIZE, N, q, tw, t)
    for p in plans(q, tw):
        out = torch.full((count, k, N), -7, dtype=torch.int32, device=DEV)
        p.matvec_shared(out, torch.from_numpy(A).to(DEV), torch.from_numpy(s).to(DEV), k, l)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), exp)


def seeded_pair(p, k, l, prng, q_bits, seed, y, transpose):
    """(rand_product_shared(seed), rand_product with the seed repeated) on device tensors."""
    count = y.shape[0]
    t1 = torch.full((count, k, N), -7, dtype=torch.int32, device=DEV)
    t2 = torch.full((count, k, N), -9, dtype=torch.int32, device=DEV)
    p.rand_product_shared(t1, y, seed, prng, q_bits, k, l, transpose)
    p.rand_product(t2, y, seed.unsqueeze(0).expand(count, seed.shape[0]).contiguous(), prng, q_bits, k, l, transpose)
    torch.cuda.synchronize()
    return t1, t2


@pytest.mark.parametrize("prng", [sc.PRNG_CHACHA, sc.PRNG_AES_CTR_DRBG])
@pytest.mark.parametrize("q,tw,k,l,q_bits,transposes", [(7681, 16, 2, 2, 13, (False, True)), (7681, 16, 3, 3, 13, (False, True)),
                                                         (7681, 16, 4, 4, 13, (False, True)), (8380417, 32, 5, 4, 23, (False,)),
                                                         (8380417, 32, 6, 5, 23, (False,))])
def test_seeded_shared_equals_repeated_seed(prng, q, tw, k, l, q_bits, transposes, plans):
    """One seed for the batch against the per-seed entry point with the seed repeated; the host twin against the device
    call."""
    g = torch.Generator(device=DEV).manual_seed(prng + k)
    seed = torch.randint(0, 256, (32,), dtype=torch.uint8, device=DEV, generator=g)
    for count in (1, 37, 20000):
        y = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
        for p in plans(q, tw):
            for transpose in transposes:
                t1, t2 = seeded_pair(p, k, l, prng, q_bits, seed, y, transpose)
                assert torch.equal(t1, t2), (count, transpose)
                if count == 37:
                    th = np.full((count, k, N), -5, dtype=np.int32)
                    p.rand_product_shared_host(th, np.ascontiguousarray(y.cpu().numpy()), seed.cpu().numpy(), prng, q_bits, k, l,
                                               transpose)
                    assert np.array_equal(th, t1.cpu().numpy()), transpose


def test_seeded_shared_host_spans_several_chunks(plans):
    """The three-stream pipeline of the host twin over several chunks of y / t."""
    q, k, l = 7681, 3, 3
    p, _ = plans(q, 16)
    rng = np.random.default_rng(11)
    seed = rng.integers(0, 256, size=32).astype(np.uint8)
    count = 20000                                              # 5.6 chunks of 16 MiB of y
    y = rng.integers(-4, 5, size=(count, l, N)).astype(np.int32)
    th = np.zeros((count, k, N), dtype=np.int32)
    p.rand_product_shared_host(th, y, seed, sc.PRNG_CHACHA, 13, k, l)
    t = torch.empty((count, k, N), dtype=torch.int32, device=DEV)
    p.rand_product_shared(t, torch.from_numpy(y).to(DEV), torch.from_numpy(seed).to(DEV), sc.PRNG_CHACHA, 13, k, l)
    torch.cuda.synchronize()
    assert np.array_equal(th, t.cpu().numpy())


def test_seeded_shared_against_golden(plans):
    """rand_product_shared(rp_seeds[i], rp_y_*) row i is rp_t_*[i] (and rp_tT_kyber3_*[i]) of the fixtures generated
    from the compiled reference."""
    G = np.load(G3)
    for name, (q, tw, k, l, q_bits) in (("kyber3", (7681, 16, 3, 3, 13)), ("dil", (8380417, 32, 5, 4, 23))):
        p, _ = plans(q, tw)
        seeds, y = G["rp_seeds"], torch.from_numpy(G["rp_y_%s" % name]).to(DEV)
        for pname, prng in (("chacha", sc.PRNG_CHACHA), ("aes", sc.PRNG_AES_CTR_DRBG)):
            for i in sorted({0, 1, len(seeds) // 2, len(seeds) - 1}):
                seed = torch.from_numpy(np.ascontiguousarray(seeds[i])).to(DEV)
                for transpose in ((False, True) if name == "kyber3" else (False,)):
                    t = torch.empty((y.shape[0], k, N), dtype=torch.int32, device=DEV)
                    p.rand_product_shared(t, y, seed, prng, q_bits, k, l, transpose)
                    torch.cuda.synchronize()
                    key = "rp_tT_%s_%s" if transpose else "rp_t_%s_%s"
                    assert np.array_equal(t.cpu().numpy()[i], G[key % (name, pname)][i]), (name, pname, i, transpose)


def test_refusals(plans):
    """Null arguments, l above the limit, n = 512, the transposed 32-bit branch with l > 1."""
    p16, _ = plans(7681, 16)
    p32, _ = plans(8380417, 32)
    z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=DEV)  # noqa: E731
    seed = torch.zeros((32,), dtype=torch.uint8, device=DEV)
    lib = sc.lib()
    assert lib.scgpu_matvec_shared_batch(p16.handle, None, z(2, 2, N).data_ptr(), z(4, 2, N).data_ptr(), 2, 2, 4, None) < 0
    assert lib.scgpu_matvec_shared_batch(p16.handle, z(4, 2, N).data_ptr(), None, z(4, 2, N).data_ptr(), 2, 2, 4, None) < 0
    assert lib.scgpu_matvec_shared_batch(None, z(4, 2, N).data_ptr(), z(2, 2, N).data_ptr(), z(4, 2, N).data_ptr(), 2, 2, 4, None) < 0
    assert lib.scgpu_rand_product_csprng_shared_batch(p16.handle, z(4, 2, N).data_ptr(), z(4, 2, N).data_ptr(), None, 32,
                                                      sc.PRNG_CHACHA, 13, 2, 2, 0, 4, None) < 0
    with pytest.raises(sc.ScgpuError):
        p16.matvec_shared(z(4, 2, N), z(2, 5, N), z(4, 5, N), 2, 5)          # l = 5 on a small modulus
    with pytest.raises(sc.ScgpuError):
        p32.matvec_shared(z(4, 2, N), z(2, 9, N), z(4, 9, N), 2, 9)          # l above sh32_mv_lmax
    w, r = O.tables(12289, 512, 16)
    p512 = sc.NttPlan(512, 12289, sc.REFERENCE, w, r)
    with pytest.raises(sc.ScgpuError):
        p512.matvec_shared(torch.zeros((4, 2, 512), dtype=torch.int32, device=DEV), torch.zeros((2, 2, 512), dtype=torch.int32, device=DEV),
                           torch.zeros((4, 2, 512), dtype=torch.int32, device=DEV), 2, 2)
    with pytest.raises(sc.ScgpuError):
        p512.rand_product_shared(torch.zeros((4, 2, 512), dtype=torch.int32, device=DEV), torch.zeros((4, 2, 512), dtype=torch.int32, device=DEV),
                                 seed, sc.PRNG_CHACHA, 14, 2, 2)
    p512.close()
    with pytest.raises(sc.ScgpuError):
        p32.rand_product_shared(z(4, 5, N), z(4, 4, N), seed, sc.PRNG_CHACHA, 23, 5, 4, transpose=True)
    with pytest.raises(sc.ScgpuError):
        p32.rand_product_shared_host(np.zeros((4, 5, N), dtype=np.int32), np.zeros((4, 4, N), dtype=np.int32),
                                     np.zeros(32, dtype=np.uint8), sc.PRNG_CHACHA, 23, 5, 4, transpose=True)


@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (8380417, 32, 6, 5)])
def test_two_streams_two_matrices_one_plan(q, tw, k, l, plans):
    """Shared products with different matrices on two streams of one plan at the same time: each call has its own table."""
    p, _ = plans(q, tw)
    g = torch.Generator(device=DEV).manual_seed(21)
    count = 1 << 17
    A1 = torch.randint(0, q, (k, l, N), dtype=torch.int32, device=DEV, generator=g)
    A2 = torch.randint(0, q, (k, l, N), dtype=torch.int32, device=DEV, generator=g)
    s1 = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
    s2 = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
    e1, e2 = torch.empty((count, k, N), dtype=torch.int32, device=DEV), torch.empty((count, k, N), dtype=torch.int32, device=DEV)
    p.matvec_shared(e1, A1, s1, k, l)
    p.matvec_shared(e2, A2, s2, k, l)
    torch.cuda.synchronize()
    assert not torch.equal(e1, e2)
    st1, st2 = torch.cuda.Stream(device=DEV), torch.cuda.Stream(device=DEV)
    o1, o2 = torch.zeros_like(e1), torch.zeros_like(e2)
    for _ in range(3):
        o1.zero_()
        o2.zero_()
        torch.cuda.synchronize()
        p.matvec_shared(o1, A1, s1, k, l, stream=st1)
        p.matvec_shared(o2, A2, s2, k, l, stream=st2)
        torch.cuda.synchronize()
        assert torch.equal(o1, e1) and torch.equal(o2, e2)


@pytest.mark.parametrize("q,tw,k,l", [(7681, 16, 3, 3), (8380417, 32, 5, 4)])
def test_graph_capture_replays_the_eager_result(q, tw, k, l, plans):
    """matvec_shared captured into a CUDA graph (table scratch, preparation and batch kernels) replays to the eager bits."""
    p, _ = plans(q, tw)
    g = torch.Generator(device=DEV).manual_seed(4)
    count = 1 << 15
    A = torch.randint(0, q, (k, l, N), dtype=torch.int32, device=DEV, generator=g)
    s = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
    eager = torch.empty((count, k, N), dtype=torch.int32, device=DEV)
    p.matvec_shared(eager, A, s, k, l)
    torch.cuda.synchronize()
    out = torch.zeros_like(eager)
    graph = torch.cuda.CUDAGraph()
    st = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(st):
        with torch.cuda.graph(graph, stream=st):
            p.matvec_shared(out, A, s, k, l, stream=st)
    for _ in range(3):
        out.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
