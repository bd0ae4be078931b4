"""Samplers that no other test reaches without the compiled reference, against references built in this file.

* Micciancio-Walter bootstrap (scgpu_gauss_plan_create_mw / scgpu_gauss_mw_streams, and create_sampler(..,
  SAMPLING_MW_BOOTSTRAP, ..) with get_vector_32 / get_vector_16 / get_bootstrap_sample).  The reference below is written
  from the algorithm of mw_bootstrap.c (network :85-99 and :112-175, mw_flip_and_round :213-241, mw_round :193-211) over
  the port's word stream and the port's sigma = 16 CDF table.  Its network constants are computed exactly.  Every
  sample is compared bit for bit except those whose double centre + x * scale lies within 4 ulp of an integer (there a
  one-ulp difference of scale could move floor()).  The output law is also computed exactly and compared with 2^22
  device samples, which guards against a misreading the kernel and the restatement would share.
* Look-up-table Knuth-Yao (scgpu_gauss_plan_create_ky_fast) over tables built here from a Knuth-Yao matrix: samples
  against a table-driven restatement of gaussian_knuth_yao_fast_sample over the port's prng_var stream, and the output
  law against the exact row probabilities of the matrix.
* scgpu_gauss_streams_host (three-stream chunked pipeline) against the port and the device call.
* The first-epoch limits of the position-addressable CDF kernels (fast_path_ok in host_sampling.cu): one sample either
  side of the last request k_cdf_chacha / k_cdf_aes may serve.

The tests without the gpu mark check the references themselves and run without a device."""
import ctypes
import functools
import math
from decimal import Decimal, localcontext
from fractions import Fraction

import numpy as np
import pytest

import _oracle as O

try:
    import torch
except ImportError:                                            # the reference checks need numpy only
    torch = None

HAVE_GPU = torch is not None and torch.cuda.is_available()
DEV = "cuda:0"
PRNGS = [O.PRNG_CHACHA, O.PRNG_AES_CTR_DRBG]


def gpu_test(f):
    return pytest.mark.gpu(pytest.mark.skipif(not HAVE_GPU, reason="no CUDA device")(f))


def seeds_for(count, length=40, salt=0):
    s = np.arange(count, dtype=np.int64)[:, None]
    j = np.arange(length, dtype=np.int64)[None, :]
    return ((s * 131 + j * 7 + 3 + salt * 29 + (s * s * 17 + j * salt) % 251) & 0xFF).astype(np.uint8)


def port_words(prng, seeds, nwords):
    """The port's prng_32 stream of every seed: prng_words without building a Python script of nwords entries."""
    script = np.zeros((nwords, 2), dtype=np.int32)
    script[:, 0] = 32
    out = np.zeros((seeds.shape[0], nwords), dtype=np.uint32)
    f = O.port()._fn("prng_script")
    for sd, row in zip(np.ascontiguousarray(seeds, dtype=np.uint8), out):
        assert f(prng, sd.ctypes.data, sd.size, 0, script.ctypes.data, nwords, row.ctypes.data) == nwords
    return out


# ---- Micciancio-Walter bootstrap: exact constants ---------------------------------------------------------------------

BASE_SIGMA, ETA, MAX_SLEVELS, LOG_BASE, MW_PRECISION, MAX_FLIPS = 16, Fraction(5, 2), 4, 1, 64, 35


@functools.lru_cache(maxsize=None)
def mw_constants():
    """(z per level, k, rr * base_sigma^2, final wide sigma^2), all exact (mw_bootstrap_create, mw_bootstrap.c:112-175)."""
    wide = Fraction(BASE_SIGMA * BASE_SIGMA)
    z = []
    for _ in range(MAX_SLEVELS - 1):
        z1 = math.isqrt(math.floor(wide / (2 * ETA * ETA)))        # floor(sqrt(w)) = isqrt(floor(w))
        z2 = max(z1 - 1, 1)
        z.append((z1, z2))
        wide = (z1 * z1 + z2 * z2) * wide
    k = -((-(MW_PRECISION - MAX_FLIPS)) // LOG_BASE)
    rr = 1 + sum(Fraction(1, 4 ** (LOG_BASE * j)) for j in range(1, k))
    return tuple(z), k, rr * BASE_SIGMA * BASE_SIGMA, wide


def f32_square(sigma):
    """sigma * sigma as the float product the library forms, as an exact fraction."""
    s = np.float32(sigma)
    return Fraction(float(np.float32(s * s)))


def mw_scale(sigma):
    """sqrt((sigma^2 - rr 256) / wide) to 50 digits, rounded to the nearest double; None below the noise floor."""
    _, _, rr256, wide = mw_constants()
    v = (f32_square(sigma) - rr256) / wide
    if v < 0:
        return None
    with localcontext() as ctx:
        ctx.prec = 50
        return float((Decimal(v.numerator) / Decimal(v.denominator)).sqrt())


@functools.lru_cache(maxsize=None)
def noise_floor_sigmas():
    """(the largest float32 sigma refused, the smallest accepted): float32(sigma * sigma) against rr 256 ~ 341.33."""
    rr256 = mw_constants()[2]
    s = np.float32(math.sqrt(float(rr256)))
    while f32_square(s) >= rr256:
        s = np.nextafter(s, np.float32(0))
    while f32_square(s) < rr256:
        s = np.nextafter(s, np.float32(np.inf))
    return float(np.nextafter(s, np.float32(0))), float(s)


SIGMA_LOW, SIGMA_FIRST = noise_floor_sigmas()


@functools.lru_cache(maxsize=None)
def base_table(precision, blinding, tail):
    return O.port().cdf_table(precision, blinding, tail, 16.0)


def cdf_base(tab, x):
    """gaussian_cdf.c:536-553 over arrays: fixed halving steps keep the largest a with tab[a] < x; sign from bit 0."""
    size = tab.size
    a = np.zeros(x.shape, dtype=np.int64)
    st = size >> 1
    while st:
        b = a + st
        a = np.where((b < size) & (tab[np.minimum(b, size - 1)] < x), b, a)
        st >>= 1
    return np.where((x & 1) == 1, a, -a)


def base_samples(words, precision, tab):
    """Base CDF samples from a word array [..., m * words per sample]: a 64-bit draw is two words, high first."""
    if precision == 64:
        w = words.reshape(words.shape[:-1] + (-1, 2)).astype(np.uint64)
        return cdf_base(tab, (w[..., 0] << np.uint64(32)) | w[..., 1])
    return cdf_base(tab, words.astype(np.uint32))


def mw_words_per_sample(precision):
    wps = precision // 32
    return 8 * wps + 2 + 29 * wps


def c_div2(v):
    """C's truncating v / 2."""
    return np.where(v < 0, -((-v) // 2), v // 2)


def mw_round_steps(r):
    """mw_round(0) (mw_bootstrap.c:193-211) over base samples r [..., k]."""
    center = np.zeros(r.shape[:-1], dtype=np.int64)
    for it in range(r.shape[-1]):
        odd = center & 1
        s = np.trunc(np.float32(0.5) * odd.astype(np.float32) + r[..., it].astype(np.float32)).astype(np.int64)
        s -= (odd == 1) & (center < 0)
        center = c_div2(center) + s
    return center


def clamp_limits(sigma, tail, centre):
    """get_vector_32's integer limits (sampling.c:560-573): float32 limit = sigma * tail, truncated sums."""
    limit = np.float32(sigma) * np.float32(tail)
    c = np.float32(centre)
    return int(np.float32(-limit + c)), int(np.float32(limit + c))


def mw_reference(words, precision, blinding, tail, sigma, centres):
    """Bootstrap samples from words [s, n * W] at per-sample float32 centres [s, n] (unclamped), and the knife-edge flags."""
    (z0, z1, z2), k, _, _ = mw_constants()
    tab = base_table(precision, blinding, tail)
    wps = precision // 32
    W = mw_words_per_sample(precision)
    s, n = centres.shape
    blk = words[:, :n * W].reshape(s, n, W)
    b = base_samples(blk[..., :8 * wps], precision, tab)
    l0 = z0[0] * b[..., 0::2] + z0[1] * b[..., 1::2]
    l1 = z1[0] * l0[..., 0::2] + z1[1] * l0[..., 1::2]
    x = z2[0] * l1[..., 0] + z2[1] * l1[..., 1]
    flip = blk[..., 8 * wps:8 * wps + 2]
    assert ((flip[..., 0] != 0) | (flip[..., 1] != 0)).all()  # a zero flip draw would shift the word positions
    center = mw_round_steps(base_samples(blk[..., 8 * wps + 2:], precision, tab))
    assert center.shape[-1] == n and k == 29
    c = centres.astype(np.float32).astype(np.float64) + x.astype(np.float64) * mw_scale(sigma)
    out = (np.floor(c).astype(np.int64) + center).astype(np.int32)
    knife = np.abs(c - np.rint(c)) <= 4 * np.spacing(np.abs(c))
    return out, knife


def assert_mw_equal(got, exp, knife, what):
    ok = (got == exp) | knife
    assert ok.all(), (what, np.argwhere(~ok)[:5].tolist(), got[~ok][:5].tolist(), exp[~ok][:5].tolist())
    assert knife.sum() <= max(1, knife.size // 10**6), (what, int(knife.sum()))


# ---- the reference's own checks (no device) ---------------------------------------------------------------------------

def test_mw_constants_exact():
    z, k, rr256, wide = mw_constants()
    assert z == ((4, 3), (22, 21), (688, 687)) and k == 29
    assert rr256 == 256 * (1 + Fraction(1, 3) * (1 - Fraction(1, 4 ** 28)))
    assert wide == 256 * 25 * 925 * (688 ** 2 + 687 ** 2)
    assert abs(math.sqrt(rr256) - 18.475) < 1e-3
    # the scale is the exactly rounded double: its square brackets the exact quotient within one ulp
    for sigma in (SIGMA_FIRST, 19.0, 40.0, 215.0, 1000.0):
        sc_ = mw_scale(sigma)
        exact = (f32_square(sigma) - rr256) / wide
        lo, hi = Fraction(np.nextafter(sc_, 0)) ** 2, Fraction(np.nextafter(sc_, np.inf)) ** 2
        assert lo < exact < hi, sigma


def test_noise_floor_between_the_sigmas_used():
    rr256 = mw_constants()[2]
    assert np.nextafter(np.float32(SIGMA_LOW), np.float32(np.inf)) == np.float32(SIGMA_FIRST)
    assert f32_square(SIGMA_LOW) < rr256 < f32_square(SIGMA_FIRST)
    assert mw_scale(SIGMA_LOW) is None and 0 < mw_scale(SIGMA_FIRST) < 1e-8


@pytest.mark.parametrize("prng", PRNGS)
def test_word_order_of_64_bit_draws(prng):
    """A prng_64 is the next two words of the stream, high word first, whatever 32-bit draws came before it."""
    seed = bytes(seeds_for(1, 48, salt=7)[0])
    script = [(32, 0), (64, 0), (64, 0), (32, 0), (32, 0), (64, 0)] * 300
    assert np.array_equal(O.port().prng_script(prng, seed, script), O.port().prng_words(prng, seed, 9 * 300))


@pytest.mark.parametrize("prng", PRNGS)
@pytest.mark.parametrize("precision", [32, 64])
@pytest.mark.parametrize("blinding,tail", [(0, 13.0), (1, 13.0), (0, 2.0)])
def test_identity_network_is_the_base_sampler(prng, precision, blinding, tail):
    """With the network replaced by the identity the restatement's base samples are the port's sigma = 16 CDF sampler.
    Blinding only scales the table's sigma by 1/sqrt 2 (the table keeps its size): the port's plain sampler at that
    sigma."""
    seeds = seeds_for(5, salt=precision + blinding)
    n = 600
    words = port_words(prng, seeds, n * precision // 32)
    got = base_samples(words, precision, base_table(precision, blinding, tail))
    sigma = float(np.float32(16.0 * math.sqrt(0.5))) if blinding else 16.0
    if blinding:
        assert np.array_equal(base_table(precision, blinding, tail), O.port().cdf_table(precision, 0, tail, sigma))
    assert np.array_equal(got, O.port().gauss_streams(O.SAMPLER_CDF, precision, 0, prng, tail, sigma, seeds, n))


def test_mw_round_matches_a_scalar_reading():
    """The vectorised mw_round against a literal scalar loop over C semantics (int arithmetic, float add, truncation)."""
    rng = np.random.default_rng(3)
    r = rng.integers(-300, 301, size=(2000, 29))
    got = mw_round_steps(r)
    for row, g in zip(r, got):
        center = 0
        for smp in row:
            odd = center & 1
            s = int(np.float32(0.5 if odd else 0.0) + np.float32(smp))
            if odd and center < 0:
                s -= 1
            center = int(center / 2) + s
        assert center == g


# ---- exact law of the bootstrap output --------------------------------------------------------------------------------

def base_law(tab):
    """P(a) of the base CDF sampler for a in [-(size-1), size-1], counted exactly over the 2^w draws (sign from parity)."""
    t = [int(v) for v in tab]
    size, top = len(t), (1 << (64 if tab.dtype == np.uint64 else 32))
    assert all(t[i] <= t[i + 1] for i in range(size - 1))
    odd, even = [0] * size, [0] * size
    for a in range(size):
        lo = t[a] + 1 if a > 0 else 0               # results a: t[a] < x <= t[a + 1] (a = 0 also takes x <= t[1])
        hi = t[a + 1] if a + 1 < size else top - 1
        if hi < lo:
            continue
        ev = hi // 2 - (lo - 1) // 2 if lo > 0 else hi // 2 + 1
        even[a], odd[a] = ev, (hi - lo + 1) - ev
    assert sum(odd) + sum(even) == top
    p = np.zeros(2 * size - 1)
    for a in range(size):
        p[size - 1 + a] += odd[a] / top
        p[size - 1 - a] += even[a] / top
    return p, size - 1                              # pmf, offset of zero


def scaled_conv(p, off, q, qoff, a, b):
    """Law of a X + b Y for X ~ (p, off), Y ~ (q, qoff) independent."""
    from scipy.signal import fftconvolve
    pa = np.zeros(a * (p.size - 1) + 1)
    pa[::a] = p
    qb = np.zeros(b * (q.size - 1) + 1)
    qb[::b] = q
    r = np.clip(fftconvolve(pa, qb), 0, None)
    return r / r.sum(), a * off + b * qoff


@functools.lru_cache(maxsize=None)
def mw_law(precision, blinding, tail, sigma, centre):
    """Exact pmf of the unclamped bootstrap output: {value: probability} as (values, probabilities)."""
    (z0, z1, z2), k, _, _ = mw_constants()
    pb, ob = base_law(base_table(precision, blinding, tail))
    l0, o0 = scaled_conv(pb, ob, pb, ob, *z0)
    l1, o1 = scaled_conv(l0, o0, l0, o0, *z1)
    keep = np.nonzero(l1 > 1e-22)[0]
    l1, o1 = l1[keep[0]:keep[-1] + 1], o1 - keep[0]
    v = np.arange(l1.size) - o1
    F = np.concatenate([[0.0], np.cumsum(l1)])              # F[i] = P(v' < v[0] + i)
    scale = mw_scale(sigma)
    c = float(np.float32(centre))
    spread = 20 * sigma
    ks = np.arange(math.floor(c - spread), math.ceil(c + spread) + 1)
    # y = floor(c + (z20 v + z21 v') scale) <= k  <=>  v' < ((k + 1 - c) / scale - z20 v) / z21
    cdf = np.zeros(ks.size)
    for i in range(0, v.size, 2048):
        vv = v[i:i + 2048, None]
        t = ((ks[None, :] + 1 - c) / scale - z2[0] * vv) / z2[1]
        idx = np.clip(np.ceil(t).astype(np.int64) - v[0], 0, v.size)
        cdf += (l1[i:i + 2048, None] * F[idx]).sum(axis=0)
    floor_law = np.diff(np.concatenate([[0.0], cdf]))
    assert cdf[-1] > 1 - 1e-12 and floor_law[0] < 1e-12
    # mw_round(0) by dynamic programming over the 29 steps: center -> trunc(center / 2) + f(smp), with
    # f(smp) = smp for an even center, trunc(smp + 0.5) for an odd one, one less again for an odd negative one
    a = np.arange(pb.size) - ob
    f_odd = np.trunc(np.float32(0.5) + a.astype(np.float32)).astype(np.int64)
    lim = 4 * ob + 8
    R = np.zeros(2 * lim + 1)
    R[lim] = 1.0
    for _ in range(k):
        nxt = np.zeros_like(R)
        for cv in np.nonzero(R)[0]:
            cen = int(cv) - lim
            base = int(cen / 2) + lim
            if cen & 1 == 0:
                np.add.at(nxt, base + a, R[cv] * pb)
            else:
                np.add.at(nxt, base + f_odd - (1 if cen < 0 else 0), R[cv] * pb)
        R = nxt
    law = np.convolve(floor_law, R)
    vals = np.arange(law.size) + ks[0] - lim
    return vals, law / law.sum()


def test_mw_law_moments():
    """The exact law's variance against sigma^2 and its mean against the centre.  The fractional part of c is dropped
    (floor), not rounded at random, so the mean sits about 1/2 below the centre whatever the centre is."""
    for centre in (3.0, -7.5):
        vals, p = mw_law(64, 0, 13.0, 40.0, centre)
        mean = float((vals * p).sum())
        var = float(((vals - mean) ** 2 * p).sum())
        assert abs(mean - (centre - 0.5125)) < 0.001, (centre, mean)
        # Measured: mean - centre = -0.5125 and var - sigma^2 = -8.26 at both centres.  The network and the floor give
        # sigma^2 - rr 256 + 1/12; mw_round(0) adds 333.0 where the design budgets rr 256 = 341.3, because an odd centre
        # adds trunc(0.5 + smp) of a zero-centred sample instead of a sample centred on 1/2.
        assert abs(var - 1600.0 + 8.26) < 0.02, (centre, var)


# ---- look-up-table Knuth-Yao: tables built from a Knuth-Yao matrix ------------------------------------------------------

def ky_matrix(rows, cols, sigma):
    """pmat[r][c] = bit c + 1 after the binary point of P(|x| = r), truncated: P(0) ~ rho(0), P(r) ~ 2 rho(r)."""
    with localcontext() as ctx:
        ctx.prec = 60
        rho = [(Decimal(-r * r) / (2 * Decimal(sigma) ** 2)).exp() * (1 if r == 0 else 2) for r in range(rows)]
        z = sum(rho)
        m = [int(p / z * (Decimal(2) ** cols)) for p in rho]
    return np.array([[(mi >> (cols - 1 - c)) & 1 for c in range(cols)] for mi in m], dtype=np.uint8)


def ddg_walk(pmat, dist, bits, col0):
    """The Knuth-Yao walk over columns col0.. with the given bits, bottom row first: ('hit', row) or ('miss', dist)."""
    for i, bit in enumerate(bits):
        dist = 2 * dist + bit
        for row in range(pmat.shape[0] - 1, -1, -1):
            dist -= int(pmat[row, col0 + i])
            if dist < 0:
                return "hit", row
    return "miss", dist


def ky_fast_tables(rows, cols, sigma, m1, m2):
    """(lut1, lut2, pmat, dist1_mask, dist2_mask) in the encoding sample_ky_fast reads (gauss.cu): lut1 maps the first
    byte to a row (bit 4 clear) or 16 | distance after 8 columns; lut2[(byte & 0x1F) + 32 distance] to a row (bit 5
    clear) or 32 | distance after 13 columns; the masks must cover every distance that occurs.  Column j of a lut
    takes bit j of its byte."""
    pmat = ky_matrix(rows, cols, sigma)
    lut1, d1 = np.zeros(256, np.uint8), []
    for b in range(256):
        kind, v = ddg_walk(pmat, 0, [(b >> j) & 1 for j in range(8)], 0)
        assert v < 16
        lut1[b] = v if kind == "hit" else 16 | v
        if kind == "miss":
            d1.append(v)
    assert max(d1) <= m1
    lut2, d2 = np.zeros(32 * (m1 + 1), np.uint8), []
    for dist in range(m1 + 1):
        for b in range(32):
            kind, v = ddg_walk(pmat, dist, [(b >> j) & 1 for j in range(5)], 8)
            if kind == "miss" and dist in d1:
                d2.append(v)
            assert kind == "miss" or v < 32
            lut2[b + 32 * dist] = v if kind == "hit" else 32 | (v & 31)
    assert max(d2) <= m2
    return lut1, lut2, pmat, m1, m2


KY_SHAPES = {"55x109": (55, 109, 3.6, 0x7, 0xF), "24x14": (24, 14, 2.2, 0x3, 0x7)}


@functools.lru_cache(maxsize=None)
def ky_tables(shape):
    return ky_fast_tables(*KY_SHAPES[shape])


class WordStream:
    """The port's word stream with prng_var's bit buffer (prng.c:1017-1048) and whole-word draws beside it."""

    def __init__(self, words):
        self.w, self.i, self.buf, self.bits = words, 0, 0, 0

    def next32(self):
        v = int(self.w[self.i])
        self.i += 1
        return v

    def var(self, n):
        ret = self.buf
        if self.bits < n:
            need = n - self.bits
            ret = (ret << need) & 0xFFFFFFFF
            self.buf = self.next32()
            ret |= self.buf & ((1 << need) - 1)
            self.buf >>= need
            self.bits = 32 - need
        else:
            self.buf >>= n
            self.bits -= n
        return ret & ((1 << n) - 1)


def ky_fast_sample(t, rs):
    """gaussian_knuth_yao_fast_sample (gaussian_knuth_yao_fast.c:303-368), table driven."""
    lut1, lut2, pmat, m1, m2 = t
    s = int(lut1[rs.var(8) & 0xFF])
    if not s & 16:
        s &= 0xF
        return -s if rs.var(1) else s
    dist = s & m1
    s = int(lut2[(rs.var(8) & 0x1F) + 32 * dist])
    if not s & 0x20:
        s &= 0x1F
        return -s if rs.var(1) else s
    dist = s & m2
    for col in range(13, pmat.shape[1]):
        dist = 2 * dist + rs.var(1)
        for row in range(pmat.shape[0] - 1, -1, -1):
            dist -= int(pmat[row, col])
            if dist < 0:
                return -row if rs.var(1) else row
    return 0


def vector_calls(draw, rs, n, calls, centre, discard, blinding):
    """sampling.c:68-145, 211-228: NORMAL or SHUFFLE vectors with discard, `calls` times on one stream."""
    thresh = {0: 0, 2: 1 << 28, 4: 1 << 30, 6: 1 << 31}[discard]
    out = []
    for _ in range(calls):
        v = [0] * n
        if blinding == O.NORMAL_SAMPLES:
            i = 0
            while i < n:
                v[i] = draw() + centre
                if not (thresh and rs.next32() < thresh):
                    i += 1
        else:
            v[0] = draw()
            i = 1
            while i < n:
                rem = 0xFFFFFFFF % i
                while True:
                    y = rs.next32()
                    if y < 0xFFFFFFFF - rem:
                        break
                j = y % i
                if j != i:
                    v[i] = v[j]
                v[j] = draw() + centre
                if not (thresh and rs.next32() < thresh):
                    i += 1
        out += v
    return out


def ky_fast_reference(t, prng, seeds, n, calls=1, centre=0, discard=0, blinding=0):
    out = np.zeros((seeds.shape[0], n * calls), dtype=np.int32)
    for s, sd in enumerate(seeds):
        nw = 4 * n * calls + 256
        while True:
            rs = WordStream(O.port().prng_words(prng, sd.tobytes(), nw))
            try:
                out[s] = vector_calls(lambda: ky_fast_sample(t, rs), rs, n, calls, centre, discard, blinding)
                break
            except IndexError:
                nw *= 2
    return out


def ky_fast_law(t):
    """Exact P(x) of the sampler: row r at column c has probability pmat[r][c] 2^-(c+1), the sign is a fair bit and
    an exhausted walk returns 0."""
    pmat = t[2]
    rows, cols = pmat.shape
    pr = [sum(Fraction(int(pmat[r, c]), 2 ** (c + 1)) for c in range(cols)) for r in range(rows)]
    law = {0: pr[0] + (1 - sum(pr))}
    for r in range(1, rows):
        law[r] = law[-r] = pr[r] / 2
    return law


def test_ky_fast_tables():
    """The shapes used: 55 x 109 with masks 0x7 / 0xF, and the smallest matrix the library takes (14 columns).  The
    look-up tables reproduce the plain walk for every 13-bit input, and the matrix rows sum to at most 1."""
    assert ky_tables("55x109")[2].shape == (55, 109) and ky_tables("55x109")[3:] == (0x7, 0xF)
    assert ky_tables("24x14")[2].shape == (24, 14)
    for shape in KY_SHAPES:
        lut1, lut2, pmat, m1, m2 = ky_tables(shape)
        assert sum(ky_fast_law(ky_tables(shape)).values()) == 1
        for b in range(1 << 13):
            bits = [(b >> j) & 1 for j in range(8)] + [(b >> (8 + j)) & 1 for j in range(5)]
            kind, v = ddg_walk(pmat, 0, bits, 0)
            e = int(lut1[b & 0xFF])
            if not e & 16:
                assert (kind, v) == ("hit", e & 0xF)
                continue
            e = int(lut2[(b >> 8) + 32 * (e & m1)])
            assert (kind, v) == (("hit", e & 0x1F) if not e & 0x20 else ("miss", e & m2))


# ---- device helpers ---------------------------------------------------------------------------------------------------

def dev_seeds(seeds):
    return torch.from_numpy(np.ascontiguousarray(seeds)).to(DEV)


def mw_gpu(plan, prng, seeds, n, sigma, centre, centres=None):
    out = torch.full((seeds.shape[0], n), 0x5A5A5A5A, dtype=torch.int32, device=DEV)
    dc = None if centres is None else torch.from_numpy(np.ascontiguousarray(centres, dtype=np.float32)).to(DEV)
    plan.mw_streams(prng, dev_seeds(seeds), n, out, sigma, centre, centres=dc)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@functools.lru_cache(maxsize=None)
def mw_plan(precision, blinding, tail):
    import libsafecrypto_b200 as sc
    return sc.GaussPlan(sc.SAMPLER_CDF, precision, blinding, tail, 0.0, mw=True)


MW_CASES = [  # (sigma, centre)
    (SIGMA_FIRST, 0.0), (SIGMA_FIRST, -7.625), (19.0, 0.5), (19.0, -0.5), (19.0, 0.75), (19.0, -0.75),
    (40.0, 0.0), (40.0, 1000.5), (215.0, -7.625), (215.0, 2.0 ** 23 - 0.5), (1000.0, -(2.0 ** 23 - 0.5)),
    (1000.0, 0.3),
]


@gpu_test
@pytest.mark.parametrize("prng", PRNGS)
@pytest.mark.parametrize("precision", [64, 32])
@pytest.mark.parametrize("blinding", [0, 1])
def test_mw_streams_against_the_reference(prng, precision, blinding):
    """Every (sigma, centre) case at tails 13 and 2 (at tail 2 the base table has 32 entries and the clamp bites; centre
    +-0.75 puts both limits on truncations toward zero that rounding would move), for 1, 33 and 130 streams and n = 1,
    77 and 300; then per-sample centres full of integers and halves."""
    W = mw_words_per_sample(precision)
    for tail in (13.0, 2.0):
        plan = mw_plan(precision, blinding, tail)
        for i, (sigma, centre) in enumerate(MW_CASES):
            count, n = (33, 77) if sigma == 19.0 else ((1, 300), (33, 77), (130, 1))[i % 3]
            seeds = seeds_for(count, salt=i + 40 * precision + 3 * blinding)
            words = port_words(prng, seeds, n * W)
            exp, knife = mw_reference(words, precision, blinding, tail, sigma, np.full((count, n), centre, np.float32))
            lo, hi = clamp_limits(sigma, tail, centre)
            exp = np.clip(exp, lo, hi)
            got = mw_gpu(plan, prng, seeds, n, sigma, centre)
            assert_mw_equal(got, exp, knife, (tail, sigma, centre, count, n))
            if tail == 2.0 and sigma == 19.0:
                assert (got == lo).any() and (got == hi).any(), (sigma, centre)
    plan = mw_plan(precision, blinding, 13.0)
    seeds = seeds_for(37, salt=5)
    rng = np.random.default_rng(precision + blinding)
    centres = (rng.integers(-400, 400, size=(37, 120)) / rng.choice([1, 2, 8], size=(37, 120))).astype(np.float32)
    centres[:, ::7] = np.float32(-2.0 ** 23 + 0.5)
    for sigma in (19.0, 215.0):
        exp, knife = mw_reference(port_words(prng, seeds, 120 * W), precision, blinding, 13.0, sigma, centres)
        assert_mw_equal(mw_gpu(plan, prng, seeds, 120, sigma, 0.0, centres=centres), exp, knife, ("centres", sigma))


@gpu_test
@pytest.mark.parametrize("prng", PRNGS)
def test_mw_streams_ragged_grid(prng):
    """129 CTAs of 128 streams plus one: the first, last and CTA-boundary streams against the reference."""
    count, n = 129 * 128 + 1, 5
    seeds = seeds_for(count, salt=77)
    plan = mw_plan(64, 0, 13.0)
    got = mw_gpu(plan, prng, seeds, n, 40.0, -7.625)
    pick = np.array([0, 1, 31, 32, 127, 128, 255, 256, 8191, 8192, 16383, 16384, count - 2, count - 1])
    exp, knife = mw_reference(port_words(prng, seeds[pick], n * mw_words_per_sample(64)), 64, 0, 13.0, 40.0,
                              np.full((pick.size, n), -7.625, np.float32))
    lo, hi = clamp_limits(40.0, 13.0, -7.625)
    assert_mw_equal(got[pick], np.clip(exp, lo, hi), knife, "ragged")


@gpu_test
def test_mw_refusals():
    import libsafecrypto_b200 as sc
    seeds = dev_seeds(seeds_for(4))
    out = torch.zeros((4, 8), dtype=torch.int32, device=DEV)
    plan = mw_plan(64, 0, 13.0)
    plan.mw_streams(O.PRNG_CHACHA, seeds, 8, out, SIGMA_FIRST, 0.0)
    for sigma in (SIGMA_LOW, 10.0, 0.0):
        with pytest.raises(sc.ScgpuError):
            plan.mw_streams(O.PRNG_CHACHA, seeds, 8, out, sigma, 0.0)
    with pytest.raises(sc.ScgpuError):
        plan.mw_streams(1, seeds, 8, out, 40.0, 0.0)                           # a generator not on the GPU path
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_CDF, 64, 0, 13.0, 16.0).mw_streams(O.PRNG_CHACHA, seeds, 8, out, 40.0, 0.0)
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_CDF, 128, 0, 13.0, 0.0, mw=True)


def dropin_lib():
    import libsafecrypto_b200 as sc
    L = sc.lib()
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
    L.get_vector_16.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_float]
    L.get_bootstrap_sample.argtypes = [ctypes.c_void_p, ctypes.c_float, ctypes.c_float]
    L.get_bootstrap_sample.restype = ctypes.c_int32
    L.get_sample.argtypes = [ctypes.c_void_p]
    L.get_sample.restype = ctypes.c_int32
    L.destroy_sampler.argtypes = [ctypes.POINTER(ctypes.c_void_p)]
    return L


@gpu_test
@pytest.mark.parametrize("prng", PRNGS)
@pytest.mark.parametrize("precision,blinding,tail", [(64, 0, 13.0), (32, 1, 2.0)])
def test_mw_dropin_sequence(prng, precision, blinding, tail):
    """create_sampler(CDF, .., SAMPLING_MW_BOOTSTRAP): get_vector_32 (clamped), prng_32, get_bootstrap_sample at varying
    sigma and centre, get_sample of the base sampler, get_vector_16 (int16 wrap past 32767), get_vector_32 again, on one
    context; the reference replays the same draws through prng_script."""
    L = dropin_lib()
    seed = bytes(((i * 11 + 5 + precision) & 0xFF) for i in range(48))
    sigma, n = 150.0, 256
    ctx = L.prng_create(5, prng, 0, 0x00100000)                                # SC_ENTROPY_USER_PROVIDED
    assert ctx and L.prng_set_entropy(ctx, seed, len(seed)) == 0 and L.prng_init(ctx, b"SAFEcrypto nonce", 16) == 0
    smp = L.create_sampler(0, precision, blinding, n, 1, ctx, tail, sigma)      # SAMPLING_MW_BOOTSTRAP = 1
    assert smp
    v1 = np.zeros(n, dtype=np.int32)
    L.get_vector_32(smp, v1.ctypes.data, n, 2.75)
    word = L.prng_32(ctx)
    boots = ((33.5, 0.25), (SIGMA_FIRST, -3.5), (500.0, 17.125), (20.0, 1e4), (1000.0, -0.75))
    singles = [L.get_bootstrap_sample(smp, sg, ce) for sg, ce in boots]
    base = L.get_sample(smp)
    v16 = np.zeros(100, dtype=np.int16)
    L.get_vector_16(smp, v16.ctypes.data, 100, 32600.5)
    v2 = np.zeros(77, dtype=np.int32)
    L.get_vector_32(smp, v2.ctypes.data, 77, -0.5)
    h = ctypes.c_void_p(smp)
    assert L.destroy_sampler(ctypes.byref(h)) == 0
    L.prng_destroy(ctx)

    d = 64 if precision == 64 else 32
    one = [(d, 0)] * 8 + [(64, 0)] + [(d, 0)] * 29
    script = one * n + [(32, 0)] + one * len(boots) + [(d, 0)] + one * 100 + one * 77
    raw = O.port().prng_script(prng, seed, script)
    W = mw_words_per_sample(precision)
    pos = 0

    def take(k):
        nonlocal pos
        pos += k
        return raw[pos - k:pos]

    def vec(m, sg, ce):
        out, knife = mw_reference(take(m * W)[None, :], precision, blinding, tail, sg, np.full((1, m), ce, np.float32))
        assert not knife.any()
        return out[0]

    lo, hi = clamp_limits(sigma, tail, 2.75)
    assert np.array_equal(v1, np.clip(vec(n, sigma, 2.75), lo, hi))
    assert word == int(take(1)[0])
    for (sg, ce), got in zip(boots, singles):
        s = int(vec(1, sg, ce)[0])
        limit = np.float32(sg) * np.float32(tail)          # get_bootstrap_sample compares in float (sampling.c:519-538)
        if np.float32(s) < np.float32(-limit + np.float32(ce)):
            s = int(np.float32(-limit + np.float32(ce)))
        if np.float32(s) > np.float32(limit + np.float32(ce)):
            s = int(np.float32(limit + np.float32(ce)))
        assert got == s, (sg, ce)
    assert base == int(base_samples(take(precision // 32), precision, base_table(precision, blinding, tail))[0])
    lo, hi = clamp_limits(sigma, tail, 32600.5)
    e16 = np.clip(vec(100, sigma, 32600.5), lo, hi)
    assert (e16 > 32767).any() and np.array_equal(v16, e16.astype(np.int16))
    lo, hi = clamp_limits(sigma, tail, -0.5)
    assert np.array_equal(v2, np.clip(vec(77, sigma, -0.5), lo, hi))
    assert pos == raw.size


def g_test(counts, probs, min_expected=20.0):
    """G statistic and p-value of observed counts against a law; cells with a small expectation are pooled."""
    from scipy.stats import chi2
    counts, probs = np.asarray(counts, np.float64), np.asarray(probs, np.float64)
    total = counts.sum()
    exp = probs * total
    big = exp >= min_expected
    obs_c = np.concatenate([counts[big], [counts[~big].sum()]])
    exp_c = np.concatenate([exp[big], [exp[~big].sum()]])
    if exp_c[-1] < min_expected:
        obs_c[-2] += obs_c[-1]
        exp_c[-2] += exp_c[-1]
        obs_c, exp_c = obs_c[:-1], exp_c[:-1]
    nz = obs_c > 0
    g = 2.0 * float((obs_c[nz] * np.log(obs_c[nz] / exp_c[nz])).sum())
    return g, float(chi2.sf(g, exp_c.size - 1))


@gpu_test
@pytest.mark.parametrize("centre", [3.0, -7.5])
def test_mw_output_law(centre):
    """2^22 samples at sigma = 40 against the exact law of mw_law (fixed seeds: deterministic)."""
    plan = mw_plan(64, 0, 13.0)
    seeds = np.random.default_rng(17).integers(0, 256, size=(4096, 40)).astype(np.uint8)
    got = mw_gpu(plan, O.PRNG_CHACHA, seeds, 1025, 40.0, centre)[:, 1:]   # a ChaCha20 stream opens with 3 zero words
    vals, p = mw_law(64, 0, 13.0, 40.0, centre)
    assert got.min() >= vals[0] and got.max() <= vals[-1]
    counts = np.bincount((got.ravel() - vals[0]).astype(np.int64), minlength=vals.size)
    g, pv = g_test(counts, p)
    assert pv > 1e-6, (centre, g, pv)


# ---- look-up-table Knuth-Yao on the device ---------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def ky_plan(shape):
    import libsafecrypto_b200 as sc
    return sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, 0, 0.0, 0.0, ky_fast=ky_tables(shape))


def ky_gpu(shape, prng, seeds, n, calls=1, centre=0, discard=0, blinding=0):
    import libsafecrypto_b200 as sc
    t = ky_tables(shape)
    plan = ky_plan(shape) if blinding == 0 else sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, blinding, 0.0, 0.0, ky_fast=t)
    out = torch.full((seeds.shape[0], n * calls), 99, dtype=torch.int32, device=DEV)
    plan.streams(prng, dev_seeds(seeds), n, out, calls=calls, centre=centre, discard=discard)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@gpu_test
@pytest.mark.parametrize("prng", PRNGS)
@pytest.mark.parametrize("shape", list(KY_SHAPES))
def test_ky_fast_against_the_reference(prng, shape):
    t = ky_tables(shape)
    for count, n, calls, centre, discard, blinding in ((1, 300, 2, 0, 0, O.NORMAL_SAMPLES), (33, 200, 2, 5, 4, O.NORMAL_SAMPLES),
                                                       (130, 64, 1, -3, 0, O.SHUFFLE_SAMPLES), (33, 77, 2, 1, 2, O.SHUFFLE_SAMPLES)):
        seeds = seeds_for(count, salt=count + calls)
        got = ky_gpu(shape, prng, seeds, n, calls, centre, discard, blinding)
        exp = ky_fast_reference(t, prng, seeds, n, calls, centre, discard, blinding)
        assert np.array_equal(got, exp), (count, n, calls, centre, discard, blinding)


@gpu_test
@pytest.mark.parametrize("shape", list(KY_SHAPES))
def test_ky_fast_output_law(shape):
    seeds = np.random.default_rng(23).integers(0, 256, size=(2048, 40)).astype(np.uint8)
    got = ky_gpu(shape, O.PRNG_AES_CTR_DRBG, seeds, 1024)
    law = ky_fast_law(ky_tables(shape))
    vals = np.array(sorted(law))
    assert got.min() >= vals[0] and got.max() <= vals[-1]
    counts = np.bincount(got.ravel() - vals[0], minlength=vals.size)
    g, pv = g_test(counts, [float(law[v]) for v in vals])
    assert pv > 1e-6, (shape, g, pv)


@gpu_test
def test_ky_fast_refusals():
    import libsafecrypto_b200 as sc
    lut1, lut2, pmat, m1, m2 = ky_tables("55x109")
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, 0, 0.0, 0.0, ky_fast=(lut1, lut2, pmat[:, :13], m1, m2))
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, 0, 0.0, 0.0, ky_fast=(lut1, lut2[:32 * (m1 + 1) - 1], pmat, m1, m2))
    with pytest.raises(sc.ScgpuError):
        sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, O.BLINDING_SAMPLES, 0.0, 0.0, ky_fast=(lut1, lut2, pmat, m1, m2))
    sc.GaussPlan(sc.SAMPLER_KNUTH_YAO_FAST, 64, 0, 0.0, 0.0, ky_fast=(lut1, lut2[:32 * (m1 + 1)], pmat[:, :14], m1, m2))


# ---- scgpu_gauss_streams_host ---------------------------------------------------------------------------------------

CHUNK_BYTES = 32 << 20


def host_buffer(shape, pinned):
    if pinned:
        return torch.full(shape, 0x7B7B7B7B, dtype=torch.int32).pin_memory().numpy()
    return np.full(shape, 0x7B7B7B7B, dtype=np.int32)


@gpu_test
@pytest.mark.parametrize("prng", PRNGS)
def test_streams_host_chunks(prng):
    """One chunk, exactly three, and four with a one-row tail (rows per chunk = 32 MiB / (4 n calls)), pageable and
    pinned output, for the fast-path request and a sequential one; against the port and the device call."""
    import libsafecrypto_b200 as sc
    n, calls = 1 << 19, 2
    rows = CHUNK_BYTES // (4 * n * calls)
    assert rows == 8
    for (blinding, discard), count, pinned in (((0, 0), 3, False), ((0, 0), 3 * rows, True), ((0, 0), 3 * rows + 1, False),
                                               ((2, 0), 3 * rows + 1, True)):
        plan = sc.GaussPlan(sc.SAMPLER_CDF, 64, blinding, 13.42, 215.0)
        seeds = seeds_for(count, salt=count)
        out = host_buffer((count, n * calls), pinned)
        plan.streams_host(prng, seeds, n, out, calls=calls, centre=-2, discard=discard)
        exp = O.port().gauss_streams(O.SAMPLER_CDF, 64, blinding, prng, 13.42, 215.0, seeds, n, centre=-2, calls=calls,
                                     discard=discard)
        assert np.array_equal(out, exp), (blinding, count, pinned)
        if count == 3 * rows + 1:
            dev = torch.empty((count, n * calls), dtype=torch.int32, device=DEV)
            plan.streams(prng, dev_seeds(seeds), n, dev, calls=calls, centre=-2, discard=discard)
            torch.cuda.synchronize()
            assert np.array_equal(dev.cpu().numpy(), out)


@gpu_test
@pytest.mark.parametrize("prng", PRNGS)
def test_streams_host_sequential_requests(prng):
    """Requests the throughput kernels do not serve: shuffle, discard, Knuth-Yao, Bernoulli, 128 rows of 32 KiB per
    chunk through two chunks and a tail; and nstreams = 0 leaves the output alone."""
    import libsafecrypto_b200 as sc
    n, calls = 4096, 2
    count = 2 * (CHUNK_BYTES // (4 * n * calls)) + 3
    seeds = seeds_for(count, salt=3)
    for sampler, blinding, discard, pinned in ((O.SAMPLER_CDF, 2, 0, False), (O.SAMPLER_CDF, 0, 4, True),
                                               (O.SAMPLER_KNUTH_YAO, 0, 0, True), (O.SAMPLER_BERNOULLI, 0, 0, False)):
        m = n if sampler == O.SAMPLER_CDF else 64
        sd = seeds if sampler == O.SAMPLER_CDF else seeds[:40]
        plan = sc.GaussPlan(sampler, 64, blinding, 13.42, 215.0)
        out = host_buffer((sd.shape[0], m * calls), pinned)
        plan.streams_host(prng, sd, m, out, calls=calls, centre=7, discard=discard)
        exp = O.port().gauss_streams(sampler, 64, blinding, prng, 13.42, 215.0, sd, m, centre=7, calls=calls, discard=discard)
        assert np.array_equal(out, exp), (sampler, blinding, discard)
    plan = sc.GaussPlan(sc.SAMPLER_CDF, 64, 0, 13.42, 215.0)
    out = host_buffer((2, 16), False)
    assert sc.lib().scgpu_gauss_streams_host(plan.handle, prng, seeds.ctypes.data, 40, 0, 8, 2, 0, 0, out.ctypes.data) == 0
    assert (out == 0x7B7B7B7B).all()


# ---- first-epoch limits of the throughput kernels -------------------------------------------------------------------

def kernels_run(fn):
    """The sampler kernels the profiler saw fn() launch, and the number of launches the library counted.  The profiler
    can lose a kernel record, so a kernel's presence is asserted only where nothing else tells the kernels apart."""
    import libsafecrypto_b200 as sc
    from torch.profiler import ProfilerActivity, profile
    before = sc.launch_count()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return {k for k in ("k_cdf_chacha", "k_cdf_aes", "k_drbg_setup", "k_stream_seq") if any(k in nm for nm in names)}, \
        sc.launch_count() - before


@gpu_test
@pytest.mark.parametrize("prng,precision,last_fast", [(O.PRNG_CHACHA, 64, 131071), (O.PRNG_CHACHA, 32, 262142),
                                                      (O.PRNG_AES_CTR_DRBG, 64, 8388608), (O.PRNG_AES_CTR_DRBG, 32, 16777216)])
def test_first_epoch_limits(prng, precision, last_fast):
    """n calls = the last sample count inside the first reseed epoch (ChaCha20: 262142 words; AES-CTR-DRBG: 4194304
    blocks) and one more: every sample against the port, and the kernel that ran.  The AES-CTR-DRBG fast path is two
    launches (k_drbg_setup, k_cdf_aes) and the sequential path one, which the library's launch counter shows; ChaCha20
    takes one launch either way, so there the profiler names the kernel."""
    import libsafecrypto_b200 as sc
    plan = sc.GaussPlan(sc.SAMPLER_CDF, precision, 0, 13.42, 215.0)
    seeds = seeds_for(2, salt=precision)
    for per, fast in ((last_fast, True), (last_fast + 1, False)):
        calls = 2 if per % 2 == 0 else 1
        n = per // calls
        out = torch.empty((2, per), dtype=torch.int32, device=DEV)
        ran, launches = kernels_run(lambda: plan.streams(prng, dev_seeds(seeds), n, out, calls=calls, centre=1))
        if prng == O.PRNG_CHACHA:
            assert launches == 1 and ran == ({"k_cdf_chacha"} if fast else {"k_stream_seq"}), (per, ran)
        else:
            assert launches == (2 if fast else 1), (per, launches)
            assert ran <= ({"k_drbg_setup", "k_cdf_aes"} if fast else {"k_stream_seq"}), (per, ran)
        exp = O.port().gauss_streams(O.SAMPLER_CDF, precision, 0, prng, 13.42, 215.0, seeds, n, centre=1, calls=calls)
        assert np.array_equal(out.cpu().numpy(), exp), per
