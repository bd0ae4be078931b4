"""ctypes binding of libscgpu.so (include/scgpu.h).  Plumbing only: pointers in, status out."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

# safecrypto_ntt_e (reference src/utils/arith/ntt.h:106-123)
REFERENCE, BARRETT, FP, AVX, SOLINAS_7681, SOLINAS_8380417 = range(6)
(OP_FWD, OP_INV, OP_FWD_LARGE, OP_INV_LARGE, OP_FFT, OP_FFT_LARGE, OP_PW, OP_PW16, OP_NORMALIZE,
 OP_CENTER, OP_POLYMUL, OP_TRIPLE16, OP_MODN, OP_MULN, OP_SQRN, OP_FLIP, OP_INVERT, OP_DIV,
 OP_PWR, OP_SCALAR, OP_SPARSE32, OP_SPARSE16) = range(22)
PRNG_AES_CTR_DRBG, PRNG_CHACHA = 0, 2
PLAN_INPUTS_IN_RANGE = 1
SAMPLER_CDF, SAMPLER_KNUTH_YAO, SAMPLER_BERNOULLI, SAMPLER_KNUTH_YAO_FAST = 0, 1, 5, 6
NORMAL_SAMPLES, BLINDING_SAMPLES, SHUFFLE_SAMPLES = 0, 1, 2


class ScgpuError(RuntimeError):
    pass


def lib_path():
    return os.path.join(_HERE, "libscgpu.so")


_lib = None


def lib():
    """Load libscgpu.so.  Fails loudly: there is no other implementation to fall back to."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not os.path.exists(path):
            raise ScgpuError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(make -C libsafecrypto_b200/csrc). No CPU fallback exists." % path)
        L = ctypes.CDLL(path)
        vp, sz, i32, u32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int32, ctypes.c_uint32
        L.scgpu_last_error.restype = ctypes.c_char_p
        L.scgpu_launch_count.restype = ctypes.c_uint64
        L.scgpu_int_peak_gops.restype = ctypes.c_double
        L.scgpu_int_peak_gops.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int]
        L.scgpu_ntt_plan_create.argtypes = [ctypes.POINTER(vp), vp, ctypes.c_int, vp, vp, ctypes.c_int, ctypes.c_int]
        L.scgpu_ntt_plan_destroy.argtypes = [vp]
        L.scgpu_ntt_plan_destroy.restype = None
        L.scgpu_ntt_plan_set_flags.argtypes = [vp, ctypes.c_uint]
        L.scgpu_gauss_cdf_table_high.argtypes = [vp, sz, ctypes.POINTER(sz), ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float]
        L.scgpu_ntt_batch.argtypes = [vp, ctypes.c_int, vp, vp, vp, sz, sz, i32, vp, vp]
        L.scgpu_ntt_batch_host.argtypes = [vp, ctypes.c_int, vp, vp, vp, sz, sz, i32, vp]
        L.scgpu_polymul_batch.argtypes = [vp, vp, vp, vp, sz, sz, vp]
        L.scgpu_polymul_batch_host.argtypes = [vp, vp, vp, vp, sz, sz]
        L.scgpu_ntt_mul_key_batch.argtypes = [vp, vp, vp, vp, ctypes.c_int, sz, sz, vp]
        L.scgpu_matvec_batch.argtypes = [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_rand_product_csprng_batch.argtypes = [vp, vp, vp, vp, sz, ctypes.c_int, u32, ctypes.c_int, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_rand_product_csprng_batch_host.argtypes = [vp, vp, vp, vp, sz, ctypes.c_int, u32, ctypes.c_int, ctypes.c_int, ctypes.c_int, sz]
        L.scgpu_matvec_shared_batch.argtypes = [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_polymul_add_batch.argtypes = [vp, vp, vp, vp, sz, vp, sz, vp]
        L.scgpu_ntt_mul_key_add_batch.argtypes = [vp, vp, vp, vp, ctypes.c_int, sz, vp, sz, vp]
        L.scgpu_matvec_add_batch.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_matvec_shared_add_batch.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_rand_product_csprng_shared_batch.argtypes = [vp, vp, vp, vp, sz, ctypes.c_int, u32, ctypes.c_int, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_rand_product_csprng_shared_batch_host.argtypes = [vp, vp, vp, vp, sz, ctypes.c_int, u32, ctypes.c_int, ctypes.c_int, ctypes.c_int, sz]
        L.scgpu_rand_matrix_csprng_batch.argtypes = [vp, vp, sz, ctypes.c_int, i32, u32, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, sz, vp]
        L.scgpu_ntt_plans_create_all.argtypes = [ctypes.POINTER(vp), ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_int]
        L.scgpu_polymul_batch_host_multi.argtypes = [ctypes.POINTER(vp), ctypes.c_int, vp, vp, vp, sz, sz]
        L.scgpu_ntt_batch_host_multi.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, vp, vp, vp, sz, sz, i32, vp]
        L.scgpu_gauss_plan_create_ky_fast.argtypes = [ctypes.POINTER(vp), vp, vp, sz, vp, ctypes.c_int, ctypes.c_int, u32, u32,
                                                      ctypes.c_int, ctypes.c_int]
        L.scgpu_gauss_plan_create_mw.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int]
        L.scgpu_gauss_mw_streams.argtypes = [vp, ctypes.c_int, vp, sz, sz, sz, ctypes.c_float, ctypes.c_float, vp, vp, vp]
        L.scgpu_gauss_plan_create_table.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, vp, sz, ctypes.c_int]
        L.scgpu_gauss_plan_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              ctypes.c_float, ctypes.c_float, ctypes.c_int]
        L.scgpu_gauss_plan_destroy.argtypes = [vp]
        L.scgpu_gauss_plan_destroy.restype = None
        L.scgpu_gauss_streams.argtypes = [vp, ctypes.c_int, vp, sz, sz, sz, sz, i32, u32, vp, vp]
        L.scgpu_gauss_streams_host.argtypes = [vp, ctypes.c_int, vp, sz, sz, sz, sz, i32, u32, vp]
        L.scgpu_prng_words.argtypes = [ctypes.c_int, vp, sz, sz, sz, sz, vp, vp]
        L.scgpu_force_montgomery.argtypes = [ctypes.c_int]
        L.scgpu_ntt_canonical_batch.argtypes = [vp, ctypes.c_int, vp, vp, sz, vp]
        L.scgpu_ntt_canonical_batch_host.argtypes = [vp, ctypes.c_int, vp, vp, sz]
        L.scgpu_set_fixed_probe_search.argtypes = [ctypes.c_int]
        L.scgpu_set_fixed_probe_search.restype = ctypes.c_int
        L.scgpu_set_fast_arith.argtypes = [ctypes.c_int]
        L.scgpu_set_fast_arith.restype = ctypes.c_int
        L.init_reduce.argtypes = [vp, sz, i32]
        L.init_reduce.restype = None
        _lib = L
    return _lib


def _check(status, what):
    if status < 0:
        raise ScgpuError("%s: %s (status %d)" % (what, lib().scgpu_last_error().decode(), status))
    return status


def launch_count():
    return int(lib().scgpu_launch_count())


def int_peak_gops(kind, iters=4096, device=0):
    return float(lib().scgpu_int_peak_gops(kind, iters, device))


PARAMS_SIZE = 60   # sizeof(ntt_params_t), packed (reference src/utils/arith/ntt.h:91-103)


def make_params(n, q):
    """A reference-layout ntt_params_t filled by the library's init_reduce()."""
    buf = ctypes.create_string_buffer(64)
    lib().init_reduce(buf, n, q)
    return buf


def _ptr(t):
    """Device or host pointer of a torch tensor / numpy array / None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def _stream_handle(stream):
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    return stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream)


class NttPlan:
    """scgpu_ntt_plan_t: one (q, n, variant) parameter set with the caller's w / r tables."""

    def __init__(self, n, q, variant, w=None, r=None, device=0, params=None):
        self.n, self.q, self.variant = n, q, variant
        self.params = params if params is not None else make_params(n, q)
        tw_bits = 0
        self._w = self._r = None
        if w is not None:
            w = np.ascontiguousarray(w)
            tw_bits = 16 if w.dtype == np.int16 else 32
            self._w = w
            if r is not None:
                self._r = np.ascontiguousarray(r, dtype=w.dtype)
        self.tw_bits = tw_bits
        h = ctypes.c_void_p()
        _check(lib().scgpu_ntt_plan_create(ctypes.byref(h), self.params, variant, _ptr(self._w), _ptr(self._r),
                                           tw_bits, device), "scgpu_ntt_plan_create")
        self.handle = h
        self.device = device

    def set_flags(self, flags):
        """scgpu_ntt_plan_set_flags (PLAN_INPUTS_IN_RANGE: the fused product skips its range vote)."""
        return _check(lib().scgpu_ntt_plan_set_flags(self.handle, int(flags)), "scgpu_ntt_plan_set_flags")

    def close(self):
        if getattr(self, "handle", None):
            lib().scgpu_ntt_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- device buffers (torch CUDA tensors) -------------------------------------------------------
    def batch(self, op, out, a, b=None, b_stride=None, count=None, scalar=0, rc=None, stream=None):
        if count is None:
            count = a.shape[0] if a.dim() > 1 else 1
        if b_stride is None:
            b_stride = 0 if (b is None or b.dim() == 1) else b.shape[-1]
        return _check(lib().scgpu_ntt_batch(self.handle, op, _ptr(out), _ptr(a), _ptr(b), b_stride, count,
                                            int(scalar), _ptr(rc), _stream_handle(stream)), "scgpu_ntt_batch")

    def polymul(self, out, a, b, count=None, stream=None):
        if count is None:
            count = a.shape[0]
        b_stride = 0 if b.dim() == 1 else b.shape[-1]
        return _check(lib().scgpu_polymul_batch(self.handle, _ptr(out), _ptr(a), _ptr(b), b_stride, count,
                                                _stream_handle(stream)), "scgpu_polymul_batch")

    def ntt_canonical(self, out, a, inverse=False, count=None, stream=None):
        if count is None:
            count = a.shape[0]
        return _check(lib().scgpu_ntt_canonical_batch(self.handle, 1 if inverse else 0, _ptr(out), _ptr(a), count,
                                                      _stream_handle(stream)), "scgpu_ntt_canonical_batch")

    def mul_key(self, out, t, key, count=None, stream=None):
        if count is None:
            count = t.shape[0]
        key_bits = key.element_size() * 8
        key_stride = 0 if key.dim() == 1 else key.shape[-1]
        return _check(lib().scgpu_ntt_mul_key_batch(self.handle, _ptr(out), _ptr(t), _ptr(key), key_bits, key_stride,
                                                    count, _stream_handle(stream)), "scgpu_ntt_mul_key_batch")

    def matvec(self, out, A, s, k, l, count=None, stream=None):
        if count is None:
            count = s.shape[0]
        return _check(lib().scgpu_matvec_batch(self.handle, _ptr(out), _ptr(A), _ptr(s), k, l, count,
                                               _stream_handle(stream)), "scgpu_matvec_batch")

    def matvec_shared(self, out, A, s, k, l, count=None, stream=None):
        """matvec with ONE matrix A [k, l, n] for every instance of s [count, l, n]."""
        if count is None:
            count = s.shape[0]
        return _check(lib().scgpu_matvec_shared_batch(self.handle, _ptr(out), _ptr(A), _ptr(s), k, l, count,
                                                      _stream_handle(stream)), "scgpu_matvec_shared_batch")

    # ---- the products above with an addend e laid out like out: out = (product + e) mod q; out may be e ----------
    def polymul_add(self, out, a, b, e, count=None, stream=None):
        if count is None:
            count = a.shape[0]
        b_stride = 0 if b.dim() == 1 else b.shape[-1]
        return _check(lib().scgpu_polymul_add_batch(self.handle, _ptr(out), _ptr(a), _ptr(b), b_stride, _ptr(e), count,
                                                    _stream_handle(stream)), "scgpu_polymul_add_batch")

    def mul_key_add(self, out, t, key, e, count=None, stream=None):
        if count is None:
            count = t.shape[0]
        key_bits = key.element_size() * 8
        key_stride = 0 if key.dim() == 1 else key.shape[-1]
        return _check(lib().scgpu_ntt_mul_key_add_batch(self.handle, _ptr(out), _ptr(t), _ptr(key), key_bits, key_stride,
                                                        _ptr(e), count, _stream_handle(stream)), "scgpu_ntt_mul_key_add_batch")

    def matvec_add(self, out, A, s, e, k, l, count=None, stream=None):
        if count is None:
            count = s.shape[0]
        return _check(lib().scgpu_matvec_add_batch(self.handle, _ptr(out), _ptr(A), _ptr(s), _ptr(e), k, l, count,
                                                   _stream_handle(stream)), "scgpu_matvec_add_batch")

    def matvec_shared_add(self, out, A, s, e, k, l, count=None, stream=None):
        """matvec_add with ONE matrix A [k, l, n] for every instance of s [count, l, n]."""
        if count is None:
            count = s.shape[0]
        return _check(lib().scgpu_matvec_shared_add_batch(self.handle, _ptr(out), _ptr(A), _ptr(s), _ptr(e), k, l, count,
                                                          _stream_handle(stream)), "scgpu_matvec_shared_add_batch")

    def rand_product(self, out, y, seeds, prng_type, q_bits, k, l, transpose=False, count=None, stream=None):
        """create_rand_product_{16,32}_csprng with the matrix sampled on the device from seeds [count, seed_len]."""
        if count is None:
            count = y.shape[0]
        return _check(lib().scgpu_rand_product_csprng_batch(self.handle, _ptr(out), _ptr(y), _ptr(seeds), seeds.shape[-1], prng_type,
                                                            q_bits, k, l, 1 if transpose else 0, count, _stream_handle(stream)),
                      "scgpu_rand_product_csprng_batch")

    def rand_product_host(self, out, y, seeds, prng_type, q_bits, k, l, transpose=False, count=None):
        if count is None:
            count = y.shape[0]
        return _check(lib().scgpu_rand_product_csprng_batch_host(self.handle, _ptr(out), _ptr(y), _ptr(seeds), seeds.shape[-1],
                                                                 prng_type, q_bits, k, l, 1 if transpose else 0, count),
                      "scgpu_rand_product_csprng_batch_host")

    def rand_product_shared(self, out, y, seed, prng_type, q_bits, k, l, transpose=False, count=None, stream=None):
        """rand_product with ONE seed [seed_len] (the key's rho) for every instance: the matrix is drawn once."""
        if count is None:
            count = y.shape[0]
        return _check(lib().scgpu_rand_product_csprng_shared_batch(self.handle, _ptr(out), _ptr(y), _ptr(seed), seed.shape[-1],
                                                                   prng_type, q_bits, k, l, 1 if transpose else 0, count,
                                                                   _stream_handle(stream)), "scgpu_rand_product_csprng_shared_batch")

    def rand_product_shared_host(self, out, y, seed, prng_type, q_bits, k, l, transpose=False, count=None):
        if count is None:
            count = y.shape[0]
        return _check(lib().scgpu_rand_product_csprng_shared_batch_host(self.handle, _ptr(out), _ptr(y), _ptr(seed), seed.shape[-1],
                                                                        prng_type, q_bits, k, l, 1 if transpose else 0, count),
                      "scgpu_rand_product_csprng_shared_batch_host")

    # ---- host buffers (numpy arrays or pinned torch CPU tensors) -----------------------------------
    def batch_host(self, op, out, a, b=None, b_stride=None, count=None, scalar=0, rc=None):
        if count is None:
            count = a.shape[0] if len(a.shape) > 1 else 1
        if b_stride is None:
            b_stride = 0 if (b is None or len(b.shape) == 1) else b.shape[-1]
        return _check(lib().scgpu_ntt_batch_host(self.handle, op, _ptr(out), _ptr(a), _ptr(b), b_stride, count,
                                                 int(scalar), _ptr(rc)), "scgpu_ntt_batch_host")

    def ntt_canonical_host(self, out, a, inverse=False, count=None):
        if count is None:
            count = a.shape[0]
        return _check(lib().scgpu_ntt_canonical_batch_host(self.handle, 1 if inverse else 0, _ptr(out), _ptr(a), count),
                      "scgpu_ntt_canonical_batch_host")

    def polymul_host(self, out, a, b, count=None):
        if count is None:
            count = a.shape[0]
        b_stride = 0 if len(b.shape) == 1 else b.shape[-1]
        return _check(lib().scgpu_polymul_batch_host(self.handle, _ptr(out), _ptr(a), _ptr(b), b_stride, count),
                      "scgpu_polymul_batch_host")


class NttPlanSet:
    """One plan per device of this process (scgpu_ntt_plans_create_all) for the *_host_multi entry points."""

    def __init__(self, n, q, variant, w, r, max_devices=64):
        self.params = make_params(n, q)
        w = np.ascontiguousarray(w)
        r = np.ascontiguousarray(r, dtype=w.dtype)
        self._w, self._r = w, r
        self.handles = (ctypes.c_void_p * max_devices)()
        got = lib().scgpu_ntt_plans_create_all(self.handles, max_devices, self.params, variant, _ptr(w), _ptr(r),
                                               16 if w.dtype == np.int16 else 32)
        _check(got, "scgpu_ntt_plans_create_all")
        self.ndev = got
        self.n = n

    def polymul_host(self, out, a, b, ndev=None):
        b_stride = 0 if len(b.shape) == 1 else b.shape[-1]
        return _check(lib().scgpu_polymul_batch_host_multi(self.handles, ndev or self.ndev, _ptr(out), _ptr(a), _ptr(b), b_stride,
                                                           a.shape[0]), "scgpu_polymul_batch_host_multi")

    def batch_host(self, op, out, a, b=None, scalar=0, rc=None, ndev=None):
        b_stride = 0 if (b is None or len(b.shape) == 1) else b.shape[-1]
        return _check(lib().scgpu_ntt_batch_host_multi(self.handles, ndev or self.ndev, op, _ptr(out), _ptr(a), _ptr(b), b_stride,
                                                       a.shape[0], int(scalar), _ptr(rc)), "scgpu_ntt_batch_host_multi")

    def close(self):
        for i in range(getattr(self, "ndev", 0)):
            if self.handles[i]:
                lib().scgpu_ntt_plan_destroy(self.handles[i])
                self.handles[i] = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def rand_matrix(A, seeds, prng_type, q, q_bits, n, k, l, transpose=False, stream=None):
    """The k x l matrix of every instance, ring by ring as uniform_random_ring_q_csprng draws it: A [count, k, l, n]."""
    return _check(lib().scgpu_rand_matrix_csprng_batch(_ptr(A), _ptr(seeds), seeds.shape[-1], prng_type, q, q_bits, n, k, l,
                                                       1 if transpose else 0, seeds.shape[0], _stream_handle(stream)),
                  "scgpu_rand_matrix_csprng_batch")


class GaussPlan:
    """scgpu_gauss_plan_t: sampler tables (built on the host with the reference's formulas) on the device."""

    def __init__(self, sampler, precision, blinding, tail, sigma, device=0, table=None, ky_fast=None, mw=False):
        h = ctypes.c_void_p()
        if mw:
            # Micciancio-Walter bootstrap over a CDF base sampler of sigma 16 (sigma argument unused)
            _check(lib().scgpu_gauss_plan_create_mw(ctypes.byref(h), precision, blinding, tail, device), "scgpu_gauss_plan_create_mw")
        elif ky_fast is not None:
            # (lut1, lut2, pmat [rows, cols], dist1_mask, dist2_mask): gaussian_knuth_yao_fast.c's constants, caller supplied
            lut1, lut2, pmat, d1, d2 = ky_fast
            lut1, lut2, pmat = (np.ascontiguousarray(x, dtype=np.uint8) for x in (lut1, lut2, pmat))
            _check(lib().scgpu_gauss_plan_create_ky_fast(ctypes.byref(h), _ptr(lut1), _ptr(lut2), lut2.size, _ptr(pmat), pmat.shape[0],
                                                         pmat.shape[1], d1, d2, blinding, device), "scgpu_gauss_plan_create_ky_fast")
        elif table is not None:
            # 128 / 192 / 256-bit CDF over a caller-built table: numpy uint64 [entries, precision / 64]
            t = np.ascontiguousarray(table, dtype=np.uint64)
            assert t.ndim == 2 and t.shape[1] * 64 == precision
            _check(lib().scgpu_gauss_plan_create_table(ctypes.byref(h), precision, blinding, ctypes.c_void_p(t.ctypes.data),
                                                       ctypes.c_size_t(t.shape[0]), device), "scgpu_gauss_plan_create_table")
        else:
            _check(lib().scgpu_gauss_plan_create(ctypes.byref(h), sampler, precision, blinding, tail, sigma, device),
                   "scgpu_gauss_plan_create")
        self.handle = h

    def close(self):
        if getattr(self, "handle", None):
            lib().scgpu_gauss_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def streams(self, prng_type, seeds, n, out, calls=1, centre=0, discard=0, stream=None):
        nstreams, seed_len = seeds.shape
        return _check(lib().scgpu_gauss_streams(self.handle, prng_type, _ptr(seeds), seed_len, nstreams, n, calls,
                                                centre, discard, _ptr(out), _stream_handle(stream)),
                      "scgpu_gauss_streams")

    def mw_streams(self, prng_type, seeds, n, out, sigma, centre=0.0, centres=None, stream=None):
        nstreams, seed_len = seeds.shape
        return _check(lib().scgpu_gauss_mw_streams(self.handle, prng_type, _ptr(seeds), seed_len, nstreams, n, sigma, centre,
                                                   _ptr(centres), _ptr(out), _stream_handle(stream)), "scgpu_gauss_mw_streams")

    def streams_host(self, prng_type, seeds, n, out, calls=1, centre=0, discard=0):
        nstreams, seed_len = seeds.shape
        return _check(lib().scgpu_gauss_streams_host(self.handle, prng_type, _ptr(seeds), seed_len, nstreams, n,
                                                     calls, centre, discard, _ptr(out)), "scgpu_gauss_streams_host")
