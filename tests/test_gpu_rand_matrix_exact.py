"""The on-device matrix sampler of the module products (scgpu_rand_matrix_csprng_batch, and through it
scgpu_rand_product_csprng_batch, its _shared_batch form and both _host twins) against a self-contained reference.

uniform_random_ring_q_csprng (module_lwe.c:519-535) fills a ring from 512 bytes of prng_mem read as little-endian UINT16,
masked to q_bits, with one conditional subtraction of q; create_csprng (:914-940) makes a fresh generator over the seed
with a 16 MiB reseed period, and the rings of a k x l matrix are drawn one after the other (i-major, or j-major into
A[i][j] for the transposed products).  ref_matrix() restates that on the port's prng_mem (oracle/sc_oracle_prng.c, pinned
to the reference by test_oracle_golden.py), so nothing the GPU computes appears on the expected side.

The tests without the gpu mark check the restatement: it reproduces the committed reference products of golden_v3.npz,
the ChaCha20 framing's three leading zero words, the seed read as a ring buffer, and the DRBG counter taken from the
seed's first word.  The gpu tests compare whole matrices bit for bit for every generator kernel (ChaCha20 with the
keystream cached in shared memory or recomputed, the two-kernel AES path and its grid-stride loop, the one-warp AES
kernel), at the largest instance the launcher accepts, with other masks, seed lengths, batch sizes and DRBG counters
that wrap, and the four product entry points across their device chunks and host pipeline chunks."""
import functools

import numpy as np
import pytest

import _oracle as O
from test_gpu_module_exact import forward, product

try:
    import torch
except ImportError:                                            # the reference checks need numpy only
    torch = None

HAVE_GPU = torch is not None and torch.cuda.is_available()
DEV = "cuda:0"
N = 256
SEED_PERIOD = 0x01000000                                       # create_csprng, module_lwe.c:921
SCGPU_OK, SCGPU_ERR_ARG, SCGPU_ERR_UNSUPPORTED = 0, -1, -3
INT32_MIN, INT32_MAX = -2**31, 2**31 - 1


def gpu_test(f):
    return pytest.mark.gpu(pytest.mark.skipif(not HAVE_GPU, reason="no CUDA device")(f))


# ---- the reference ---------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def draws(prng, seed, rings):
    """The UINT16 stream of a fresh create_csprng generator over `seed` (bytes): `rings` rows of 512 bytes of prng_mem."""
    words = O.port().prng_script(prng, seed, [(4, 512)] * rings, seed_period=SEED_PERIOD)
    v = words.view("<u2").reshape(rings, N)
    v.flags.writeable = False
    return v


def ref_matrix(prng, seed, q, q_bits, k, l, transpose):
    """A [k, l, n] of one instance: ring r is A[r / l][r % l], or A[r % k][r / k] when transposed."""
    x = draws(prng, bytes(seed), k * l).astype(np.int64) & (0xFFFFFFFF if q_bits >= 32 else (1 << q_bits) - 1)
    x -= np.where(x >= q, q, 0)
    A = x.reshape(l, k, N).transpose(1, 0, 2) if transpose else x.reshape(k, l, N)
    return np.ascontiguousarray(A, dtype=np.int32)


def ref_matrices(prng, seeds, q, q_bits, k, l, transpose):
    return np.stack([ref_matrix(prng, s, q, q_bits, k, l, transpose) for s in seeds])


def counter_seed(c, tail):
    """A DRBG seed whose generator starts at counter c: instantiation leaves 3 ^ le32(seed[0:4]) (ctr_drbg.c:100-147)."""
    return np.concatenate([np.frombuffer(((c ^ 3) & 0xFFFFFFFF).to_bytes(4, "little"), np.uint8), tail])


# ---- which kernel each case reaches ----------------------------------------------------------------------------------
# route() restates launch_gen_rings (rand_product.cu) for n = 256:
#   ChaCha20                                  -> k_gen_rings<CHACHA20>: one warp per instance, each lane k l keystream
#                                                blocks; kept in shared memory between the two passes when k l <= 24,
#                                                computed a second time otherwise
#   AES-CTR-DRBG, SCGPU_GEN_AES_WARP=1        -> k_gen_rings<AES>: one warp per instance
#   AES-CTR-DRBG                              -> k_gen_setup_aes + k_gen_rings_aes: one block per thread, a grid of at
#                                                most one 1024-thread CTA per SM striding over count * 32 k l blocks
GENS = ["chacha", "aes", "aes-warp"]
GEN_PRNG = {"chacha": O.PRNG_CHACHA, "aes": O.PRNG_AES_CTR_DRBG, "aes-warp": O.PRNG_AES_CTR_DRBG}
GEN_LAUNCHES = {"chacha": 1, "aes": 2, "aes-warp": 1}
SMS = 148


def route(gen, k, l, count, sms=SMS):
    if gen == "chacha":
        return "k_gen_rings<CHACHA20>, keystream %s" % ("cached" if k * l <= 24 else "recomputed")
    if gen == "aes-warp":
        return "k_gen_rings<AES>"
    items = count * 32 * k * l
    grid = min(sms, -(-items // 1024))
    return "k_gen_setup_aes + k_gen_rings_aes, %d pass(es)" % -(-items // (grid * 1024))


# (k, l) around the ChaCha20 cache limit k l = 24 and up to the largest Dilithium set
SHAPES = [(1, 1), (2, 2), (3, 3), (4, 4), (5, 4), (4, 6), (5, 5), (6, 5), (8, 8)]
# k l = 32767: the largest instance below the 16 MiB reseed period (k l 512 bytes per instance)
LARGEST = [(1, 32767), (181, 181)]
# (q, q_bits): the Kyber, NewHope-sized and Dilithium readings, a mask above q (16 bits leave entries up to
# 65535 - q), a mask below q (no subtraction ever) and the 32-bit mask
MODULI = [(7681, 13), (12289, 14), (8380417, 23), (7681, 16), (12289, 12), (7681, 32), (8380417, 32)]
SEED_LENS = [1, 3, 4, 31, 32, 33, 36, 39, 40, 41, 48, 64]
# 4 instances per CTA of the one-warp kernels; 1100 Kyber k = 3 instances are 316800 AES blocks, > 148 * 1024
COUNTS = [1, 3, 4, 5, 129, 1100]
DRBG_SHAPE = (2, 3)


def drbg_counters(k, l):
    """Counter starts whose blocks reach 2^32 - 1 or wrap: the last block of the third is 0xFFFFFFFF, the fourth wraps on
    its last block."""
    return [2**32 - 1, 2**32 - 5, 2**32 - 32 * k * l, 2**32 - 32 * k * l + 1]


def case_routes():
    """The route of every (generator, k, l, count) the matrix tests below launch."""
    got = set()
    for gen in GENS:
        cases = [(k, l, 5) for k, l in SHAPES] + [(k, l, 1) for k, l in LARGEST] + [(2, 3, 5), (3, 2, 7)] + \
                [(3, 3, c) for c in COUNTS] + [DRBG_SHAPE + (4,)]
        got.update(route(gen, k, l, c) for k, l, c in cases)
    return got


def test_cases_reach_every_route():
    routes = case_routes()
    for want in ("k_gen_rings<CHACHA20>, keystream cached", "k_gen_rings<CHACHA20>, keystream recomputed", "k_gen_rings<AES>",
                 "k_gen_setup_aes + k_gen_rings_aes, 1 pass(es)"):
        assert want in routes, want
    assert any(r.startswith("k_gen_setup_aes") and not r.endswith(" 1 pass(es)") for r in routes), routes


# ---- the reference against fixtures and against the framing ------------------------------------------------------------

def test_reference_reproduces_the_golden_products():
    """The restated matrix through the exact product gives the reference's own create_rand_product_{16,32}_csprng output
    (golden_v3.npz, both generators, Kyber k = 3 both draw orders, Dilithium (5, 4)): ring order, byte order, mask,
    subtraction and the transposed destination."""
    G = O.golden("golden_v3")
    seeds = G["rp_seeds"]
    for name, (q, tw, k, l, q_bits, transposes) in (("kyber3", (7681, 16, 3, 3, 13, (False, True))),
                                                      ("dil", (8380417, 32, 5, 4, 23, (False,)))):
        Fy = forward(q, tw, G["rp_y_%s" % name])
        for pname, prng in (("chacha", O.PRNG_CHACHA), ("aes", O.PRNG_AES_CTR_DRBG)):
            for transpose in transposes:
                key = "rp_%s_%s_%s" % ("tT" if transpose else "t", name, pname)
                A = ref_matrices(prng, seeds, q, q_bits, k, l, transpose)
                assert np.array_equal(product(q, tw, A, Fy), G[key]), key


def test_chacha_stream_starts_with_three_zero_words():
    """The ChaCha20-CSPRNG framing emits three zero words before the first keystream word (chacha20_csprng.c:72-84); a
    64-bit draw is stored low word first, so coefficients 0-3 and 6-7 of an instance's first ring are 0 before masking,
    4-5 are not."""
    rng = np.random.default_rng(11)
    seeds = [bytes(32), bytes([255]) * 32] + [rng.integers(0, 256, 32, dtype=np.uint8).tobytes() for _ in range(6)]
    for seed in seeds:
        v = draws(O.PRNG_CHACHA, seed, 2)
        assert not v[0, [0, 1, 2, 3, 6, 7]].any(), seed.hex()
        assert v[0, 4:6].any() and v[0, 8:].any() and v[1].any(), seed.hex()
        assert draws(O.PRNG_AES_CTR_DRBG, seed, 1)[0, :8].any(), seed.hex()


@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG], ids=["chacha", "aes"])
@pytest.mark.parametrize("L", [1, 3, 7, 33])
def test_seed_is_read_as_a_ring_buffer(prng, L):
    """A seed of L bytes and the same bytes repeated cyclically to 40 bytes or more give the same matrix: ChaCha20 takes
    40 bytes (key, IV), the DRBG 36 (counter word, key), both from the start of the ring buffer."""
    rng = np.random.default_rng(100 + L)
    seed = rng.integers(0, 256, L, dtype=np.uint8)
    A = ref_matrix(prng, seed, 7681, 13, 2, 3, False)
    for m in (40, 41, 48, 64):
        assert np.array_equal(ref_matrix(prng, np.resize(seed, m), 7681, 13, 2, 3, False), A), m
    other = np.resize(seed, 40)
    other[35] ^= 1                                            # a DRBG key byte, a ChaCha20 IV byte
    assert not np.array_equal(ref_matrix(prng, other, 7681, 13, 2, 3, False), A)


@pytest.mark.parametrize("c", [1, 0, 2**32 - 1, 2**32 - 5, 2**31])
def test_drbg_counter_starts_at_the_seed_word(c):
    """le32(seed[0:4]) = c ^ 3 starts the DRBG at counter c: with the key bytes equal, the stream from counter c is the
    stream from counter c - 1 (mod 2^32) one 16-byte block later, across 1 KiB refills and across the 32-bit wrap."""
    tail = np.random.default_rng(7).integers(0, 256, 36, dtype=np.uint8)
    rings = 3                                                 # 96 blocks: one refill of the 1 KiB transfer buffer
    now = draws(O.PRNG_AES_CTR_DRBG, counter_seed(c, tail).tobytes(), rings).reshape(-1)
    before = draws(O.PRNG_AES_CTR_DRBG, counter_seed((c - 1) % 2**32, tail).tobytes(), rings).reshape(-1)
    assert np.array_equal(now[:-8], before[8:])               # 8 UINT16 per block
    assert not np.array_equal(now, before)


# ---- GPU: the matrix ----------------------------------------------------------------------------------------------------

if HAVE_GPU:
    import libsafecrypto_b200 as sc
    from libsafecrypto_b200 import binding as B


@pytest.fixture(params=GENS)
def gen(request, monkeypatch):
    """The generator kernel: SCGPU_GEN_AES_WARP is read at every launch."""
    if request.param == "aes-warp":
        monkeypatch.setenv("SCGPU_GEN_AES_WARP", "1")
    else:
        monkeypatch.delenv("SCGPU_GEN_AES_WARP", raising=False)
    return request.param


@pytest.fixture(params=["aes", "aes-warp"])
def aes_gen(request, monkeypatch):
    if request.param == "aes-warp":
        monkeypatch.setenv("SCGPU_GEN_AES_WARP", "1")
    else:
        monkeypatch.delenv("SCGPU_GEN_AES_WARP", raising=False)
    return request.param


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def gpu_matrix(gen, seeds, q, q_bits, k, l, transpose):
    """rand_matrix into a buffer filled with -1; also the number of kernel launches it made."""
    seeds = np.ascontiguousarray(seeds, dtype=np.uint8)
    A = torch.full((seeds.shape[0], k, l, N), -1, dtype=torch.int32, device=DEV)
    d_seeds = torch.from_numpy(seeds).to(DEV)
    torch.cuda.synchronize()
    before = sc.launch_count()
    B.rand_matrix(A, d_seeds, GEN_PRNG[gen], q, q_bits, N, k, l, transpose)
    torch.cuda.synchronize()
    return A.cpu().numpy(), sc.launch_count() - before


def assert_matrix(got, exp, label, names=None):
    """Equal, or a message naming the instance, the matrix entry and its ring in draw order, and the coefficient."""
    if np.array_equal(got, exp):
        return
    bad = np.argwhere(got != exp)
    c, i, j, x = (int(v) for v in bad[0])
    k, l = got.shape[1], got.shape[2]
    what = " (%s)" % names[c] if names is not None else ""
    raise AssertionError(
        "%s: instance %d%s, A[%d][%d] (ring %d i-major, %d j-major), coefficient %d: got %d, expected %d; %d coefficients "
        "in %d instances and %d rings differ" % (label, c, what, i, j, i * l + j, j * k + i, x, got[c, i, j, x], exp[c, i, j, x],
                                                 len(bad), len(np.unique(bad[:, 0])), len(np.unique(bad[:, 0:3], axis=0))))


def check_matrix(gen, seeds, q, q_bits, k, l, transpose, label, names=None):
    got, launches = gpu_matrix(gen, seeds, q, q_bits, k, l, transpose)
    r = route(gen, k, l, len(seeds), sms())
    label = "%s q=%d q_bits=%d k=%d l=%d transpose=%s count=%d [%s]" % (label, q, q_bits, k, l, transpose, len(seeds), r)
    assert launches == GEN_LAUNCHES[gen], "%s: %d launches" % (label, launches)
    assert_matrix(got, ref_matrices(GEN_PRNG[gen], seeds, q, q_bits, k, l, transpose), label, names)


def random_seeds(rng, count, L):
    return rng.integers(0, 256, size=(count, L), dtype=np.uint8)


@gpu_test
@pytest.mark.parametrize("k,l", SHAPES)
def test_matrix_shapes(gen, k, l):
    """5 instances (two CTAs of the one-warp kernels), both draw orders."""
    q, q_bits = (8380417, 23) if k >= 5 else (7681, 13)
    seeds = random_seeds(np.random.default_rng(31 * k + l), 5, 32)
    for transpose in (False, True):
        check_matrix(gen, seeds, q, q_bits, k, l, transpose, gen)


@gpu_test
@pytest.mark.parametrize("k,l", LARGEST)
def test_matrix_largest_instance(gen, k, l):
    """k l = 32767 rings, 16 MiB - 512 bytes of generator output in one instance: the ChaCha20 recompute path at its
    longest per-lane run, the AES kernels at their largest block index."""
    seeds = random_seeds(np.random.default_rng(k), 1, 32)
    for transpose in (False, True):
        check_matrix(gen, seeds, 7681, 13, k, l, transpose, gen)


@gpu_test
@pytest.mark.parametrize("q,q_bits", MODULI)
def test_matrix_moduli(gen, q, q_bits):
    """Every mask reading: canonical entries, entries up to 2^16 - 1 - q after the one subtraction, no subtraction."""
    seeds = random_seeds(np.random.default_rng(q + q_bits), 5, 32)
    for transpose in (False, True):
        check_matrix(gen, seeds, q, q_bits, 2, 3, transpose, gen)
    exp = ref_matrices(GEN_PRNG[gen], seeds, q, q_bits, 2, 3, False)
    if q_bits >= 16:
        assert exp.max() >= q or q > 65535                    # the non-canonical entries are really there


@gpu_test
@pytest.mark.parametrize("L", SEED_LENS)
def test_matrix_seed_lengths(gen, L):
    """Seeds of L bytes, read as a ring buffer, at instance offsets inst * L; the all-zero and all-0xFF seeds."""
    seeds = random_seeds(np.random.default_rng(L), 7, L)
    seeds[2] = 0
    seeds[5] = 0xFF
    names = ["random"] * 7
    names[2], names[5] = "all-zero seed", "all-0xFF seed"
    for transpose in (False, True):
        check_matrix(gen, seeds, 7681, 13, 3, 2, transpose, "%s seed_len=%d" % (gen, L), names)


@gpu_test
@pytest.mark.parametrize("count", COUNTS)
def test_matrix_batch_sizes(gen, count):
    """Kyber k = 3; 1100 instances make k_gen_rings_aes stride over its grid more than once."""
    seeds = random_seeds(np.random.default_rng(count), count, 32)
    check_matrix(gen, seeds, 7681, 13, 3, 3, False, gen)


@gpu_test
def test_matrix_drbg_counter_wrap(aes_gen):
    """DRBG counters that reach 0xFFFFFFFF on the last block of an instance or wrap inside it, in one batch."""
    k, l = DRBG_SHAPE
    rng = np.random.default_rng(5)
    cs = drbg_counters(k, l)
    seeds = np.stack([counter_seed(c, rng.integers(0, 256, 28, dtype=np.uint8)) for c in cs])
    names = ["counter 0x%08X" % c for c in cs]
    for transpose in (False, True):
        check_matrix(aes_gen, seeds, 7681, 13, k, l, transpose, aes_gen, names)


def raw_rand_matrix(A_ptr, seeds, seed_len, prng, q, q_bits, n, k, l, count):
    return sc.lib().scgpu_rand_matrix_csprng_batch(A_ptr, seeds.data_ptr(), seed_len, prng, q, q_bits, n, k, l, 0, count,
                                                   torch.cuda.current_stream().cuda_stream)


@gpu_test
def test_matrix_alignment(gen):
    """The kernels store 8 and 16 bytes at a time: an A 4, 8 or 12 bytes off a 16-byte boundary is refused with
    SCGPU_ERR_ARG before anything runs; an aligned view into a larger buffer works."""
    k, l, count = 2, 3, 5
    size = count * k * l * N
    seeds = random_seeds(np.random.default_rng(9), count, 32)
    d_seeds = torch.from_numpy(seeds).to(DEV)
    buf = torch.full((size + 8,), -1, dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    for words in (1, 2, 3):
        before = sc.launch_count()
        assert raw_rand_matrix(buf.data_ptr() + 4 * words, d_seeds, 32, GEN_PRNG[gen], 7681, 13, N, k, l, count) == SCGPU_ERR_ARG
        assert sc.launch_count() == before
    torch.cuda.synchronize()
    assert bool((buf == -1).all())
    view = buf[4:4 + size].view(count, k, l, N)
    assert view.data_ptr() % 16 == 0
    B.rand_matrix(view, d_seeds, GEN_PRNG[gen], 7681, 13, N, k, l)
    torch.cuda.synchronize()
    assert_matrix(view.cpu().numpy(), ref_matrices(GEN_PRNG[gen], seeds, 7681, 13, k, l, False), "%s aligned view" % gen)
    assert bool((buf[:4] == -1).all()) and bool((buf[4 + size:] == -1).all())


# ---- GPU: the products --------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def plans():
    made = {}

    def get(q, tw, n=N):
        if (q, tw, n) not in made:
            w, r = O.tables(q, n, tw)
            made[(q, tw, n)] = sc.NttPlan(n, q, sc.REFERENCE, w, r)
        return made[(q, tw, n)]
    yield get
    for p in made.values():
        p.close()


@pytest.fixture
def auto_arith():
    old = sc.lib().scgpu_set_fast_arith(0)
    yield 0
    sc.lib().scgpu_set_fast_arith(old)


# (q, tw, q_bits, k, l, transpose)
PRODUCT_SHAPES = [(7681, 16, 13, k, k, t) for k in (2, 3, 4) for t in (False, True)] + [(8380417, 32, 23, 6, 5, False)]


def device_chunk(k, l):
    """Instances per matrix chunk of scgpu_rand_product_csprng_batch: 48 MB of scratch."""
    return (48 << 20) // (k * l * N * 4)


def host_rows(k, l):
    """Instances per chunk of the three-stream pipeline of the _host twins: 16 MB of y or t staging."""
    return (16 << 20) // max(4 * l * N, 4 * k * N)


def picked(count, step, rng):
    """First and last instance of every chunk of `step`, +-1 around each boundary, 16 random instances."""
    idx = {count - 1}
    for b in range(0, count, step):
        idx.update(range(max(0, b - 1), min(count, b + 2)))
        idx.add(min(count, b + step) - 1)
    idx.update(int(x) for x in rng.integers(0, count, size=16))
    return np.array(sorted(idx))


def assert_product(got, exp, idx, label):
    if np.array_equal(got, exp):
        return
    bad = np.argwhere(got != exp)
    c, i, x = (int(v) for v in bad[0])
    raise AssertionError("%s: instance %d, output row %d, coefficient %d: got %d, expected %d; %d of the %d compared instances "
                         "differ: %s" % (label, idx[c], i, x, got[c, i, x], exp[c, i, x], len(np.unique(bad[:, 0])), len(idx),
                                         [int(idx[v]) for v in np.unique(bad[:, 0])][:12]))


@gpu_test
@pytest.mark.parametrize("prng", [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG], ids=["chacha", "aes"])
@pytest.mark.parametrize("L", [7, 33, 48])
@pytest.mark.parametrize("q,tw,q_bits,k,l,transpose", PRODUCT_SHAPES)
def test_products_across_chunks(prng, L, q, tw, q_bits, k, l, transpose, auto_arith, plans, monkeypatch):
    """rand_product over 2 device chunks + 1 instance and rand_product_host over 3 pipeline chunks + 1, with seeds of L
    bytes at offsets off * L; rand_product_shared and rand_product_shared_host with one seed.  y is any SINT32 (default
    plan); the instances around every chunk boundary and 16 random ones are compared with ref_matrix through the exact
    product, every output must be a canonical residue."""
    monkeypatch.delenv("SCGPU_GEN_AES_WARP", raising=False)
    gen = "chacha" if prng == O.PRNG_CHACHA else "aes"
    p = plans(q, tw)
    rng = np.random.default_rng(1000 * k + 100 * l + 10 * L + prng + transpose)
    chunk, rows = device_chunk(k, l), host_rows(k, l)
    n_dev, n_host = 2 * chunk + 1, 3 * rows + 1
    top = max(n_dev, n_host)
    y = rng.integers(INT32_MIN, INT32_MAX + 1, size=(top, l, N), dtype=np.int32)
    seeds = random_seeds(rng, top, L)
    d_y, d_seeds = torch.from_numpy(y).to(DEV), torch.from_numpy(seeds).to(DEV)
    shape = "q=%d k=%d l=%d transpose=%s seed_len=%d" % (q, k, l, transpose, L)

    def expect(idx, shared):
        A = ref_matrix(prng, seeds[0], q, q_bits, k, l, transpose) if shared else \
            ref_matrices(prng, seeds[idx], q, q_bits, k, l, transpose)
        return product(q, tw, A, forward(q, tw, y[idx]))

    def check(t, count, step, shared, label):
        assert t.min() >= 0 and t.max() < q, "%s: outputs outside [0, q): %d .. %d" % (label, t.min(), t.max())
        idx = picked(count, step, rng)
        assert_product(t[idx], expect(idx, shared), idx, label)

    t = torch.full((n_dev, k, N), -7, dtype=torch.int32, device=DEV)
    p.rand_product(t, d_y[:n_dev], d_seeds[:n_dev], prng, q_bits, k, l, transpose)
    torch.cuda.synchronize()
    check(t.cpu().numpy(), n_dev, chunk, False, "%s rand_product, device chunks of %d [%s]" % (shape, chunk, route(gen, k, l, chunk, sms())))

    th = np.full((n_host, k, N), -5, dtype=np.int32)
    p.rand_product_host(th, np.ascontiguousarray(y[:n_host]), np.ascontiguousarray(seeds[:n_host]), prng, q_bits, k, l, transpose)
    check(th, n_host, rows, False, "%s rand_product_host, pipeline chunks of %d" % (shape, rows))

    t = torch.full((n_dev, k, N), -7, dtype=torch.int32, device=DEV)
    p.rand_product_shared(t, d_y[:n_dev], d_seeds[0].contiguous(), prng, q_bits, k, l, transpose)
    torch.cuda.synchronize()
    check(t.cpu().numpy(), n_dev, chunk, True, "%s rand_product_shared [%s]" % (shape, route(gen, k, l, 1)))

    th = np.full((n_host, k, N), -5, dtype=np.int32)
    p.rand_product_shared_host(th, np.ascontiguousarray(y[:n_host]), np.ascontiguousarray(seeds[0]), prng, q_bits, k, l, transpose)
    check(th, n_host, rows, True, "%s rand_product_shared_host, pipeline chunks of %d" % (shape, rows))


# ---- GPU: refusals ------------------------------------------------------------------------------------------------------

# (label, prng, seed_len, n, k, l, status)
REFUSED = [("k l = 32768", 2, 32, N, 1, 32768, SCGPU_ERR_UNSUPPORTED),
           ("k l = 32768", 0, 32, N, 128, 256, SCGPU_ERR_UNSUPPORTED),
           ("n = 512", 2, 32, 512, 2, 2, SCGPU_ERR_UNSUPPORTED),
           ("seed_len = 0", 0, 0, N, 2, 2, SCGPU_ERR_ARG),
           ("k = 0", 2, 32, N, 0, 2, SCGPU_ERR_ARG),
           ("l = 0", 0, 32, N, 2, 0, SCGPU_ERR_ARG),
           ("k = l = 0", 2, 32, N, 0, 0, SCGPU_ERR_ARG),
           ("PRNG type 1", 1, 32, N, 2, 2, SCGPU_ERR_UNSUPPORTED),
           ("PRNG type 3", 3, 32, N, 2, 2, SCGPU_ERR_UNSUPPORTED)]


@gpu_test
def test_refusals(plans):
    """Every entry point refuses, with the status of include/scgpu.h and without launching anything: an instance of
    32768 rings (it would reach the generator's 16 MiB reseed period), n != 256, an empty seed, k or l = 0, the PRNG types
    without a device generator.  k l = 32767 is accepted (test_matrix_largest_instance)."""
    L = sc.lib()
    st = torch.cuda.current_stream().cuda_stream
    count = 2
    seeds = torch.zeros((count, 32), dtype=torch.uint8, device=DEV)
    h_seeds = np.zeros((count, 32), dtype=np.uint8)
    for label, prng, seed_len, n, k, l, status in REFUSED:
        A = torch.full((count * max(k * l * n, 1),), -1, dtype=torch.int32, device=DEV)
        y = torch.zeros((count * max(l * n, 1),), dtype=torch.int32, device=DEV)
        t = torch.full((count * max(k * n, 1),), -1, dtype=torch.int32, device=DEV)
        h_y, h_t = y.cpu().numpy(), t.cpu().numpy()
        p = plans(12289, 16, 512) if n == 512 else plans(7681, 16)
        torch.cuda.synchronize()
        before = sc.launch_count()
        calls = {
            "rand_matrix": lambda: L.scgpu_rand_matrix_csprng_batch(A.data_ptr(), seeds.data_ptr(), seed_len, prng, p.q, 13, n, k, l,
                                                                    0, count, st),
            "rand_product": lambda: L.scgpu_rand_product_csprng_batch(p.handle, t.data_ptr(), y.data_ptr(), seeds.data_ptr(), seed_len,
                                                                      prng, 13, k, l, 0, count, st),
            "rand_product_shared": lambda: L.scgpu_rand_product_csprng_shared_batch(p.handle, t.data_ptr(), y.data_ptr(),
                                                                                    seeds.data_ptr(), seed_len, prng, 13, k, l, 0,
                                                                                    count, st),
            "rand_product_host": lambda: L.scgpu_rand_product_csprng_batch_host(p.handle, h_t.ctypes.data, h_y.ctypes.data,
                                                                                h_seeds.ctypes.data, seed_len, prng, 13, k, l, 0,
                                                                                count),
            "rand_product_shared_host": lambda: L.scgpu_rand_product_csprng_shared_batch_host(p.handle, h_t.ctypes.data,
                                                                                              h_y.ctypes.data, h_seeds.ctypes.data,
                                                                                              seed_len, prng, 13, k, l, 0, count),
        }
        for name, call in calls.items():
            got = call()
            assert got == status, "%s, %s: status %d, expected %d (%s)" % (name, label, got, status, L.scgpu_last_error().decode())
        torch.cuda.synchronize()
        assert sc.launch_count() == before, label
        assert bool((A == -1).all()) and bool((t == -1).all()) and bool((h_t == -1).all()), label
