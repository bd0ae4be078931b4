"""ctypes bindings for the two CPU checkers (TEST INFRASTRUCTURE ONLY).

* ``port()``  -> oracle/libscoracle.so, our plain-C restatement (oracle/sc_oracle*.c)
* ``ref()``   -> oracle/_ref/libscref.so, the unmodified reference compiled by oracle/Makefile
                 (present only when it was built in the dev container; it travels to the GPU box)

Both expose the same batch-driver calling convention (oracle/ref_driver.c, oracle/sc_oracle.h),
so a test can run one input through either.
"""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")

# safecrypto_ntt_e, /root/reference/src/utils/arith/ntt.h:106-123
REFERENCE, BARRETT, FP, AVX, SOLINAS_7681, SOLINAS_8380417 = range(6)
VARIANT_NAMES = {REFERENCE: "reference", BARRETT: "barrett", FP: "fp", AVX: "avx",
                 SOLINAS_7681: "7681", SOLINAS_8380417: "8380417"}

(OP_FWD, OP_INV, OP_FWD_LARGE, OP_INV_LARGE, OP_FFT, OP_FFT_LARGE, OP_PW, OP_PW16, OP_NORMALIZE,
 OP_CENTER, OP_POLYMUL, OP_TRIPLE16, OP_MODN, OP_MULN, OP_SQRN, OP_FLIP, OP_INVERT, OP_DIV,
 OP_PWR, OP_SCALAR, OP_SPARSE32, OP_SPARSE16) = range(22)

PRNG_AES_CTR_DRBG, PRNG_CHACHA = 0, 2
SAMPLER_CDF, SAMPLER_KNUTH_YAO, SAMPLER_BERNOULLI, SAMPLER_KNUTH_YAO_FAST = 0, 1, 5, 6
NORMAL_SAMPLES, BLINDING_SAMPLES, SHUFFLE_SAMPLES = 0, 1, 2

# (tw_bits, q, n) of build_tools/ntt_table_gen/main.c:19-37
TABLE_PARAMS = [(16, 7681, 256), (16, 12289, 512), (16, 12289, 1024), (16, 18433, 512), (16, 18433, 1024),
                (32, 4206593, 512), (32, 4206593, 1024), (32, 5767169, 512), (32, 5767169, 1024),
                (32, 8380417, 256), (32, 8399873, 512), (32, 10223617, 512), (32, 10223617, 1024),
                (32, 16813057, 512), (32, 51750913, 512), (32, 51750913, 1024), (32, 134348801, 1024)]


def _vp(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def aligned(a, dtype=None, align=64):
    """Copy into a 64-byte aligned contiguous array: the reference's AVX2 variant uses aligned
    loads on caller buffers (sc_malloc gives 32-byte alignment, safecrypto_private.c:82-96)."""
    a = np.asarray(a, dtype=dtype)
    buf = np.empty(a.nbytes + align, dtype=np.uint8)
    off = (-buf.ctypes.data) % align
    out = buf[off:off + a.nbytes].view(a.dtype).reshape(a.shape)
    out[...] = a
    return out


def script_words(kind, arg):
    """Output words of one prng_script entry (oracle/sc_oracle.h)."""
    kind, arg = int(kind), int(arg)
    return {64: 2, 128: 4, 3: 2, 6: 2, 5: 0}.get(kind, (arg + 3) // 4 if kind == 4 else 1)


class Checker:
    def __init__(self, path, prefix):
        self.lib = ctypes.CDLL(path)
        self.prefix = prefix
        self.path = path
        f = self._fn("ntt_batch")
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int] * 5 + [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                           ctypes.c_void_p, ctypes.c_int32]
        g = self._fn("gauss_streams")
        g.restype = ctypes.c_int
        g.argtypes = [ctypes.c_int] * 4 + [ctypes.c_float, ctypes.c_float, ctypes.c_uint32, ctypes.c_void_p,
                                           ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int32,
                                           ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t]
        s = self._fn("prng_script")
        s.restype = ctypes.c_int
        s.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_void_p,
                      ctypes.c_size_t, ctypes.c_void_p]
        self._fn("num_threads").restype = ctypes.c_int

    def _fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def num_threads(self):
        return int(self._fn("num_threads")())

    def ntt_batch(self, variant, op, n, q, tw_bits, a, b=None, w=None, r=None, scalar=0, threads=0,
                  want_rc=False, a_dtype=np.int32):
        a = aligned(np.asarray(a, dtype=a_dtype).reshape(-1, n))
        count = a.shape[0]
        out = aligned(np.zeros((count, n), dtype=np.int32))
        w = None if w is None else aligned(w)
        r = None if r is None else aligned(r)
        b_stride = 0
        if b is not None:
            b = aligned(b)
            # 1-D operand = one row shared by the whole batch; 2-D = one row per batch item
            b_stride = 0 if b.ndim == 1 else b.shape[-1]
        rc = np.zeros(count, dtype=np.int32)
        ret = self._fn("ntt_batch")(variant, op, n, q, tw_bits, _vp(out), _vp(a), _vp(b), b_stride,
                                    _vp(w), _vp(r), count, threads, _vp(rc), int(scalar))
        if want_rc:
            return out, rc, ret
        return out

    def prng_script(self, prng_type, seed, script, seed_period=0):
        seed = np.frombuffer(bytes(seed), dtype=np.uint8).copy()
        script = np.ascontiguousarray(script, dtype=np.int32).reshape(-1, 2)
        nout = int(sum(script_words(k, a) for k, a in script))
        out = np.zeros(nout, dtype=np.uint32)
        got = self._fn("prng_script")(prng_type, _vp(seed), seed.size, seed_period, _vp(script),
                                      script.shape[0], _vp(out))
        assert got == nout, (got, nout)
        return out

    def prng_words(self, prng_type, seed, nwords, seed_period=0):
        return self.prng_script(prng_type, seed, [(32, 0)] * nwords, seed_period)

    def cdf_table(self, precision, blinding, tail, sigma):
        f = self._fn("cdf_table")
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t]
        cap = 1 << 16
        if precision > 64:
            nw = precision // 64
            buf = np.zeros(cap * nw, dtype=np.uint64)
            size = f(precision, blinding, tail, sigma, _vp(buf), cap)
            assert 0 < size <= cap
            return buf[:size * nw].reshape(size, nw).copy()
        buf = np.zeros(cap, dtype=np.uint64 if precision == 64 else np.uint32)
        size = f(precision, blinding, tail, sigma, _vp(buf), cap)
        assert 0 < size <= cap
        return buf[:size].copy()

    def set_high_table(self, precision, table):
        """Inject a 128 / 192-bit CDF table (uint64 [entries, precision / 64]) for gauss_streams(): the port
        needs one (it does not restate the reference's multi-precision table construction), the compiled
        reference has the table it built overwritten.  None clears."""
        f = self._fn("set_high_table")
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        if table is None:
            self._high = getattr(self, "_high", {})
            self._high.pop(precision, None)
            assert f(precision, None, 0) == 0
            return
        t = np.ascontiguousarray(table, dtype=np.uint64)
        self._high = getattr(self, "_high", {})
        self._high[precision] = t                       # the reference driver keeps the pointer
        assert f(precision, _vp(t), t.shape[0]) == 0


    def ky_table(self, bitwidth, tail, sigma, blinding=0):
        bitwidth |= blinding << 12
        f = self._fn("ky_table")
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t,
                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        cap = 1 << 23
        buf = np.zeros(cap, dtype=np.uint8)
        dims = np.zeros(3, dtype=np.int32)
        sz = f(bitwidth, tail, sigma, _vp(buf), cap, dims[0:].ctypes.data, dims[1:].ctypes.data, dims[2:].ctypes.data)
        assert 0 < sz <= cap
        return buf[:sz].reshape(int(dims[0]), int(dims[1])).copy(), int(dims[2])

    def ber_table(self, tail, sigma):
        f = self._fn("ber_table")
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t,
                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        buf = np.zeros(64 * 8, dtype=np.uint8)
        dims = np.zeros(3, dtype=np.int32)
        sz = f(tail, sigma, _vp(buf), buf.size, dims[0:].ctypes.data, dims[1:].ctypes.data, dims[2:].ctypes.data)
        return buf[:sz].reshape(-1, 8).copy(), int(dims[1]), int(dims[2])

    def gauss_streams(self, sampler, precision, blinding, prng_type, tail, sigma, seeds, n, discard=0,
                      centre=0, threads=0, calls=1):
        seeds = np.ascontiguousarray(seeds, dtype=np.uint8)
        nstreams, seed_len = seeds.shape
        out = np.zeros((nstreams, calls * n), dtype=np.int32)
        fail = self._fn("gauss_streams")(sampler, precision, blinding, prng_type, tail, sigma, discard,
                                         _vp(seeds), seed_len, nstreams, n, centre, _vp(out), threads, calls)
        assert fail == 0
        return out


class RefChecker(Checker):
    """The reference library also exports its generated twiddle tables as data symbols."""

    def kyfast_tables(self, dimension):
        """(lut1, lut2, pmat [rows, cols], dist1_mask, dist2_mask) of gaussian_knuth_yao_fast_{256,512}_create, read out of
        the compiled reference."""
        f = self.lib.ref_kyfast_tables
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        lut1, lut2, pmat = np.zeros(256, np.uint8), np.zeros(4096, np.uint8), np.zeros(1 << 16, np.uint8)
        dims = np.zeros(5, np.int32)
        assert f(dimension, _vp(lut1), _vp(lut2), lut2.size, _vp(pmat), pmat.size, _vp(dims)) == 0
        rows, cols = int(dims[0]), int(dims[1])
        return lut1, lut2[:int(dims[4])].copy(), pmat[:rows * cols].reshape(rows, cols).copy(), int(dims[2]), int(dims[3])

    def mw_streams(self, prng_type, seeds, n, tail, sigma, centre=0.0, sigmas=None, centres=None, threads=0):
        """create_sampler(CDF, 64-bit, SAMPLING_MW_BOOTSTRAP) per stream; n get_vector_32 samples at (sigma, centre), or
        n get_bootstrap_sample(sigmas[s, i], centres[s, i]) calls when the arrays are given."""
        f = self.lib.ref_mw_streams
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_float, ctypes.c_float,
                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
        seeds = np.ascontiguousarray(seeds, dtype=np.uint8)
        out = np.zeros((seeds.shape[0], n), dtype=np.int32)
        per = centres is not None
        if per:
            centres = np.ascontiguousarray(centres, dtype=np.float32)
            sigmas = np.ascontiguousarray(sigmas if sigmas is not None else np.full(centres.shape, sigma), dtype=np.float32)
        else:
            centres = np.array([centre], dtype=np.float32)
        assert f(prng_type, _vp(seeds), seeds.shape[1], seeds.shape[0], n, tail, sigma, _vp(sigmas) if per else None, _vp(centres),
                 1 if per else 0, _vp(out), threads) == 0
        return out

    def rand_product(self, tw_bits, variant, n, q, q_bits, k, l, transpose, prng_type, seeds, y, w, r, want_matrix=False, threads=0):
        """create_rand_product_{16,32}_csprng (module_lwe.c:588-748) per instance, CSPRNG as create_csprng makes it.
        Returns t [count, k, n] (and the matrix in DRAW order [count, k l, n])."""
        f = self.lib.ref_rand_product
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int] * 9 + [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
        seeds = np.ascontiguousarray(seeds, dtype=np.uint8)
        count = seeds.shape[0]
        y = aligned(np.asarray(y, dtype=np.int32).reshape(count, l, n))
        t = aligned(np.zeros((count, k, n), dtype=np.int32))
        A = aligned(np.zeros((count, k * l, n), dtype=np.int32)) if want_matrix else None
        w, r = aligned(w), aligned(r)
        assert f(tw_bits, variant, n, q, q_bits, k, l, 1 if transpose else 0, prng_type, _vp(seeds), seeds.shape[1], _vp(y), _vp(t),
                 _vp(A), _vp(w), _vp(r), count, threads) == 0
        return (t, A) if want_matrix else t

    def table(self, kind, q, n, tw_bits):
        ct = ctypes.c_int16 if tw_bits == 16 else ctypes.c_int32
        size = n // 2 if kind == "inv_w" else n
        arr = (ct * size).in_dll(self.lib, "%s%d_n%d" % (kind, q, n))
        return np.ctypeslib.as_array(arr).copy()


class PortChecker(Checker):
    def roots_of_unity(self, q, n, tw_bits):
        f = self.lib.orc_roots_of_unity
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        w = np.zeros(n, dtype=np.int32)
        r = np.zeros(n, dtype=np.int32)
        g = ctypes.c_int64(0)
        assert f(q, n, _vp(w), _vp(r), ctypes.byref(g)) == 0
        dt = np.int16 if tw_bits == 16 else np.int32
        return w.astype(dt), r.astype(dt), int(g.value)

    def scalar(self, name, variant, n, q, *args):
        class P(ctypes.Structure):
            _fields_ = [("n", ctypes.c_int32), ("q", ctypes.c_int32), ("m", ctypes.c_int32), ("k", ctypes.c_int32),
                        ("inv_q_dbl", ctypes.c_double), ("inv_q_flt", ctypes.c_float)]
        p = P()
        self.lib.orc_init_reduce(ctypes.byref(p), n, q)
        f = getattr(self.lib, "orc_" + name)
        f.restype = ctypes.c_int32
        return int(f(variant, *[ctypes.c_int32(int(x)) for x in args], ctypes.byref(p)))


_cache = {}


def build_port():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "port"])


def port():
    if "port" not in _cache:
        path = os.path.join(ORACLE_DIR, "libscoracle.so")
        srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.startswith("sc_oracle")]
        if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(s) for s in srcs):
            build_port()
        _cache["port"] = PortChecker(path, "orc_")
    return _cache["port"]


def ref_available():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libscref.so"))


def ref():
    if "ref" not in _cache:
        _cache["ref"] = RefChecker(os.path.join(ORACLE_DIR, "_ref", "libscref.so"), "ref_")
    return _cache["ref"]


def golden(name):
    """Arrays of tests/golden/<name>.npz as a dict.  A fixture stores each distinct array once: its optional
    `_aliases` member lists (name, stored name) pairs for the arrays equal to one already stored."""
    with np.load(os.path.join(ROOT, "tests", "golden", name + ".npz")) as z:
        out = {k: z[k] for k in z.files}
    for alias, stored in out.pop("_aliases", np.zeros((0, 2), dtype=str)):
        out[str(alias)] = out[str(stored)]
    return out


def dedup_arrays(arrays):
    """The inverse of golden(): keep the first of each group of equal arrays, list the others in `_aliases`."""
    import hashlib
    out, seen, aliases = {}, {}, []
    for k, a in arrays.items():
        h = hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + np.ascontiguousarray(a).tobytes()).digest()
        if h in seen:
            aliases.append((k, seen[h]))
        else:
            seen[h] = k
            out[k] = a
    if aliases:
        out["_aliases"] = np.array(aliases, dtype=str)
    return out


def tables(q, n, tw_bits):
    """(w, r) for a parameter set -- from the port's generator (validated against the reference's
    generated ntt_tables.c in tests/test_oracle_vs_ref.py and tests/golden/tables.json)."""
    w, r, _ = port().roots_of_unity(q, n, tw_bits)
    return w, r


def high_precision_cdf_table(precision, tail, sigma, blinding=0):
    """What gauss_cdf_create_high_precision (gaussian_cdf.c:192-318) computes when its multi-precision floats
    are exact: entry i = floor(s_i), s_1 = d / 2, s_{i+1} = s_i + d exp(-i^2 / (2 sigma^2)),
    d = 2 / sqrt(2 pi) * 2^precision / sigma, entry 0 = 0, saturating to all-ones.  Returned as uint64
    [entries, precision / 64] with word 0 least significant.  Used as a realistic table for the sampling tests."""
    from decimal import Decimal, getcontext
    getcontext().prec = precision // 3 + 40
    entries = 1 << int(np.ceil(np.log2(np.float32(tail) * np.float32(sigma))))
    sg = Decimal(float(np.float32(sigma)))
    if blinding == 1:
        sg = sg * Decimal(0.5).sqrt()
    pi = Decimal("3.14159265358979323846264338327950288419716939937510582097494459230781640628620899862803482534211706798214808651")
    d = Decimal(2) / (2 * pi).sqrt() * (Decimal(2) ** precision) / sg
    e = -Decimal(0.5) / (sg * sg)
    nw = precision // 64
    top = (1 << precision) - 1
    tab = np.zeros((entries, nw), dtype=np.uint64)
    s = d / 2
    i = 1
    while i < entries - 1:
        v = int(s)
        if v > top:
            break
        for j in range(nw):
            tab[i, j] = (v >> (64 * j)) & 0xFFFFFFFFFFFFFFFF
        s += d * (e * i * i).exp()
        i += 1
    tab[i:, :] = np.uint64(0xFFFFFFFFFFFFFFFF)
    return tab
