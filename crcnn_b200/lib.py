"""ctypes plumbing over the C ABI in include/crcnn_b200.h (crcnn_b200/libcrcnn_b200.so).

Python is only the harness language here (tests, bench.py): every arithmetic step happens in the
CUDA kernels behind the C ABI.  There is no CPU fallback -- a missing library or a missing GPU is
an error, never a silent detour.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# CRCNN_B200_LIB selects another build of the same library (kernel A/B runs of tools/ntt_ab.py)
LIB_PATH = os.environ.get("CRCNN_B200_LIB") or os.path.join(_HERE, "libcrcnn_b200.so")

_u64p = C.POINTER(C.c_uint64)
_u32p = C.POINTER(C.c_uint32)
_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int)
_vp = C.c_void_p
_vpp = C.POINTER(C.c_void_p)

# every symbol include/crcnn_b200.h declares: (name, restype, argtypes)
_I, _L = C.c_int, C.c_long
SYMBOLS = [
    ("crcnn_last_error", C.c_char_p, [_vp]),
    ("crcnn_ctx_create", _I, [_I, _I, _u64p, C.c_uint64, _I, _vpp]),
    ("crcnn_ctx_destroy", _I, [_vp]),
    ("crcnn_ctx_set_stream", _I, [_vp, _vp]),
    ("crcnn_ctx_sync", _I, [_vp]),
    ("crcnn_ctx_alloc_stats", _I, [_vp, C.POINTER(C.c_longlong)]),
    ("crcnn_ctx_set_weight_cache_bytes", _I, [_vp, C.c_size_t]),
    ("crcnn_ctx_set_tensor_core_mode", _I, [_vp, C.c_int, C.c_int, C.c_size_t]),
    ("crcnn_ctx_set_limb_split_mode", _I, [_vp, C.c_int]),
    ("crcnn_ctx_set_limb_split_reduction", _I, [_vp, C.c_int]),
    ("crcnn_ctx_set_relin_mode", _I, [_vp, C.c_int]),
    ("crcnn_ctx_ntt_table", _I, [_vp, _I, _I, _u64p]),
    ("crcnn_ctx_bsk_count", _I, [_vp]),
    ("crcnn_tensor_upload", _I, [_vp, _vp, _L, _I, _vpp]),
    ("crcnn_tensor_upload_ex", _I, [_vp, _vp, _L, _I, _I, _vpp]),
    ("crcnn_tensor_upload_on", _I, [_vp, _vp, _L, _I, _I, _vp, _vpp]),
    ("crcnn_tensor_upload_into", _I, [_vp, _vp, _vp, _I, _vp]),
    ("crcnn_ctx_wait_stream", _I, [_vp, _vp]),
    ("crcnn_tensor_download", _I, [_vp, _vp, _vp]),
    ("crcnn_tensor_download_ex", _I, [_vp, _vp, _I, _vp]),
    ("crcnn_tensor_free", _I, [_vp, _vp]),
    ("crcnn_tensor_count", _L, [_vp]),
    ("crcnn_tensor_ct_size", _I, [_vp]),
    ("crcnn_tensor_slice", _I, [_vp, _vp, _L, _L, _vpp]),
    ("crcnn_tensor_device_ptr", _I, [_vp, _vpp, _i32p]),
    ("crcnn_tensor_wrap_alloc", _I, [_vp, _L, _I, _I, _vpp]),
    ("crcnn_plain_upload", _I, [_vp, _u64p, _L, _I, _L, _vpp]),
    ("crcnn_plain_upload_sparse", _I, [_vp, _u32p, _u64p, _u32p, _L, _vpp]),
    ("crcnn_plain_encode", _I, [_vp, _f32p, _L, _vpp]),
    ("crcnn_plain_encode_f64", _I, [_vp, C.POINTER(C.c_double), _L, _vpp]),
    ("crcnn_plain_get", _I, [_vp, _vp, _L, _u64p]),
    ("crcnn_plain_get_ntt", _I, [_vp, _vp, _L, _u64p]),
    ("crcnn_plain_free", _I, [_vp, _vp]),
    ("crcnn_plain_count", _L, [_vp]),
    ("crcnn_evk_upload", _I, [_vp, _u64p, _I, _i32p, _vpp]),
    ("crcnn_evk_free", _I, [_vp, _vp]),
    ("crcnn_conv_forward", _I, [_vp, _vp, _vp, _vp] + [_I] * 9 + [_vpp]),
    ("crcnn_conv_forward_shard", _I, [_vp, _vp, _vp, _vp] + [_I] * 11 + [_vpp]),
    ("crcnn_fc_forward", _I, [_vp, _vp, _vp, _vp, _I, _I, _I, _vpp]),
    ("crcnn_fc_forward_shard", _I, [_vp, _vp, _vp, _vp, _I, _I, _I, _I, _I, _vpp]),
    ("crcnn_pool_forward", _I, [_vp, _vp] + [_I] * 8 + [_vp, _vpp]),
    ("crcnn_bn_forward", _I, [_vp, _vp, _I, _I, _I, _I, _vp, _vp, _vpp]),
    ("crcnn_pool_bn_forward", _I, [_vp, _vp] + [_I] * 8 + [_vp, _vp, _vp, _vpp]),
    ("crcnn_pool_bn_fc_fc_forward", _I, [_vp, _vp] + [_I] * 8 + [_vp] * 7 + [_I, _I, _vpp]),
    ("crcnn_fc_fc_forward", _I, [_vp, _vp, _vp, _vp, _vp, _vp, _I, _I, _I, _I, _vpp]),
    ("crcnn_conv_pool_bn_forward", _I, [_vp, _vp, _vp, _vp] + [_I] * 13 + [_vp, _vp, _vp, _vpp]),
    ("crcnn_conv_pool_bn_forward_shard", _I, [_vp, _vp, _vp, _vp] + [_I] * 13 + [_vp, _vp, _vp, _I, _I, _vpp]),
    ("crcnn_square_forward", _I, [_vp, _vp, _vp, _vpp]),
    ("crcnn_transform_to_ntt", _I, [_vp, _vp]),
    ("crcnn_transform_from_ntt", _I, [_vp, _vp]),
    ("crcnn_plain_op", _I, [_vp, _vp, _vp, _L, _I]),
    ("crcnn_add_many", _I, [_vp, _vp, _vpp]),
    ("crcnn_square", _I, [_vp, _vp, _vpp]),
    ("crcnn_relinearize", _I, [_vp, _vp, _vp, _vpp]),
    ("crcnn_prof_enable", _I, [_vp, _I]),
    ("crcnn_prof_reset", _I, [_vp]),
    ("crcnn_prof_count", _I, [_vp]),
    ("crcnn_prof_get", _I, [_vp, _I, C.c_char_p, C.POINTER(C.c_long), C.POINTER(C.c_double)]),
    ("crcnn_prof_get_work", _I, [_vp, _I, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    ("crcnn_probe_imad", _I, [_vp, _I, _I, _I, C.POINTER(C.c_double)]),
    ("crcnn_pinned_alloc", _I, [C.c_size_t, _vpp]),
    ("crcnn_pinned_free", _I, [_vp]),
    ("crcnn_stream_create", _I, [_vp, _vpp]),
    ("crcnn_stream_destroy", _I, [_vp, _vp]),
    ("crcnn_event_create", _I, [_vp, _vpp]),
    ("crcnn_event_record", _I, [_vp, _vp, _vp]),
    ("crcnn_stream_wait_event", _I, [_vp, _vp, _vp]),
    ("crcnn_event_elapsed_ms", _I, [_vp, _vp, _vp, C.POINTER(C.c_double)]),
    ("crcnn_event_destroy", _I, [_vp, _vp]),
    ("crcnn_tensor_download_async", _I, [_vp, _vp, _vp]),
    ("crcnn_comm_unique_id", _I, [_vp]),
    ("crcnn_comm_create", _I, [_vp, _vp, _I, _I, _vpp]),
    ("crcnn_comm_destroy", _I, [_vp, _vp]),
    ("crcnn_comm_all_gather", _I, [_vp, _vp, _vp, _I, C.POINTER(C.c_long), _I, _vpp]),
    ("crcnn_keys_upload", _I, [_vp, _vp, _vp, _vpp]),
    ("crcnn_keys_free", _I, [_vp, _vp]),
    ("crcnn_decrypt", _I, [_vp, _vp, _vp, _vp]),
    ("crcnn_noise_budget", _I, [_vp, _vp, _vp, _i32p, _i32p]),
    ("crcnn_reencrypt", _I, [_vp, _vp, _vp, C.c_uint64, C.c_double, _vp, _vpp, _vp, _vp]),
    ("crcnn_encrypt_values", _I, [_vp, _vp, _f32p, C.c_long, C.c_uint64, C.c_double, _vp, _vpp]),
    ("crcnn_decrypt_values", _I, [_vp, _vp, _vp, _f32p]),
    ("crcnn_probe_pipe", _I, [_vp, _I, _I, _I, _I, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
]

_lib = None


def load():
    """Load the CUDA extension; raise (never fall back) if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "crcnn_b200/libcrcnn_b200.so is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C crcnn_b200/csrc`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class CrcnnError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("crcnn_b200 error %d: %s" % (code, msg))
        self.code = code


class Handle:
    """Owning wrapper of a device object (tensor / plain pack / evaluation keys)."""

    def __init__(self, eng, ptr, kind):
        self.eng, self.ptr, self.kind = eng, ptr, kind

    def free(self):
        if self.ptr and self.eng.h:
            getattr(self.eng.lib, "crcnn_%s_free" % self.kind)(self.eng.h, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """One context = one GPU + one stream (see include/crcnn_b200.h)."""

    def __init__(self, n, primes, t, device=0):
        self.lib = load()
        self.n, self.K, self.t = int(n), len(primes), int(t)
        self.primes = [int(p) for p in primes]
        self.stride = self.n + 1
        self.h = None
        q = np.array(self.primes, dtype=np.uint64)
        h = C.c_void_p()
        rc = self.lib.crcnn_ctx_create(self.n, self.K, q.ctypes.data_as(_u64p), self.t, device, C.byref(h))
        if rc != 0:
            raise CrcnnError(rc, self.lib.crcnn_last_error(None).decode())
        self.h = h
        self.S = self.lib.crcnn_ctx_bsk_count(self.h)

    @classmethod
    def adopt(cls, ctx_ptr, n, primes, t):
        """Engine view of a context somebody else owns (the C++ Runtime behind crcnn_b200/host.py): same C ABI calls, no destroy."""
        self = cls.__new__(cls)
        self.lib = load()
        self.n, self.K, self.t = int(n), len(primes), int(t)
        self.primes = [int(p) for p in primes]
        self.stride = self.n + 1
        self.h = C.c_void_p(ctx_ptr)
        self.owned = False
        self.S = self.lib.crcnn_ctx_bsk_count(self.h)
        return self

    def close(self):
        if self.h and getattr(self, "owned", True):
            self.lib.crcnn_ctx_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise CrcnnError(rc, self.lib.crcnn_last_error(self.h).decode())

    def _new(self, fn, kind, *args):
        out = C.c_void_p()
        self._chk(fn(self.h, *args, C.byref(out)))
        return Handle(self, out, kind)

    # ---- context
    def set_stream(self, stream_ptr):
        self._chk(self.lib.crcnn_ctx_set_stream(self.h, C.c_void_p(stream_ptr)))

    def sync(self):
        self._chk(self.lib.crcnn_ctx_sync(self.h))

    def set_weight_cache_bytes(self, b):
        self._chk(self.lib.crcnn_ctx_set_weight_cache_bytes(self.h, int(b)))

    def set_tensor_core_mode(self, mode, min_fanin=0, scratch_bytes=0):
        self._chk(self.lib.crcnn_ctx_set_tensor_core_mode(self.h, int(mode), int(min_fanin), int(scratch_bytes)))

    def set_limb_split_mode(self, mode):
        self._chk(self.lib.crcnn_ctx_set_limb_split_mode(self.h, int(mode)))

    def set_limb_split_reduction(self, mode):
        self._chk(self.lib.crcnn_ctx_set_limb_split_reduction(self.h, int(mode)))

    def set_relin_mode(self, mode):
        self._chk(self.lib.crcnn_ctx_set_relin_mode(self.h, int(mode)))

    def ntt_table(self, slot, which):
        out = np.zeros(self.n, dtype=np.uint64)
        self._chk(self.lib.crcnn_ctx_ntt_table(self.h, slot, which, out.ctypes.data_as(_u64p)))
        return out

    def ct_words(self, size=2):
        return size * self.K * self.stride

    # ---- tensors
    def upload(self, cts, size=2, ntt_form=False):
        a = np.ascontiguousarray(cts, dtype=np.uint64)
        count = a.size // self.ct_words(size)
        assert count * self.ct_words(size) == a.size, "buffer is not a whole number of ciphertexts"
        return self._new(self.lib.crcnn_tensor_upload_ex, "tensor", a.ctypes.data, count, size, int(ntt_form))

    def upload_ptr(self, host_ptr, count, size=2, ntt_form=False):
        """Upload from a raw host address (e.g. a pinned torch tensor)."""
        return self._new(self.lib.crcnn_tensor_upload_ex, "tensor", host_ptr, count, size, int(ntt_form))

    def upload_ptr_on(self, host_ptr, count, copy_stream_ptr, size=2, ntt_form=False):
        """H2D on a separate copy stream (double buffering); call wait_stream() before using the tensor."""
        return self._new(self.lib.crcnn_tensor_upload_on, "tensor", host_ptr, count, size, int(ntt_form), C.c_void_p(copy_stream_ptr))

    def upload_into(self, t, host_ptr, copy_stream_ptr=None, ntt_form=False):
        """Overwrite an existing tensor from a raw (pinned) host address through the context's staging buffer."""
        self._chk(self.lib.crcnn_tensor_upload_into(self.h, host_ptr, t.ptr, int(ntt_form), C.c_void_p(copy_stream_ptr)))

    def wait_stream(self, stream_ptr):
        self._chk(self.lib.crcnn_ctx_wait_stream(self.h, C.c_void_p(stream_ptr)))

    def download(self, t, ntt_form=False, out=None):
        count, size = self.lib.crcnn_tensor_count(t.ptr), self.lib.crcnn_tensor_ct_size(t.ptr)
        if out is None:
            out = np.empty((count, size, self.K, self.stride), dtype=np.uint64)
        self._chk(self.lib.crcnn_tensor_download_ex(self.h, t.ptr, int(ntt_form), out.ctypes.data))
        return out

    def download_ptr(self, t, host_ptr, ntt_form=False):
        self._chk(self.lib.crcnn_tensor_download_ex(self.h, t.ptr, int(ntt_form), host_ptr))

    def count(self, t):
        return self.lib.crcnn_tensor_count(t.ptr)

    def slice(self, t, first, count):
        return self._new(self.lib.crcnn_tensor_slice, "tensor", t.ptr, first, count)

    def device_ptr(self, t):
        p, f = C.c_void_p(), C.c_int()
        self._chk(self.lib.crcnn_tensor_device_ptr(t.ptr, C.byref(p), C.byref(f)))
        return p.value, f.value

    def alloc(self, count, size=2, ntt_form=False):
        return self._new(self.lib.crcnn_tensor_wrap_alloc, "tensor", count, size, int(ntt_form))

    # ---- plaintext packs / keys
    def plain_upload(self, words, coeff_count=None):
        a = np.ascontiguousarray(words, dtype=np.uint64)
        if a.ndim == 1:
            a = a[None, :]
        count, stride = a.shape
        cc = stride if coeff_count is None else coeff_count
        return self._new(self.lib.crcnn_plain_upload, "plain", a.ctypes.data_as(_u64p), count, cc, stride)

    def plain_upload_sparse(self, idx, val, offsets):
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        val = np.ascontiguousarray(val, dtype=np.uint64)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
        return self._new(self.lib.crcnn_plain_upload_sparse, "plain", idx.ctypes.data_as(_u32p),
                         val.ctypes.data_as(_u64p), offsets.ctypes.data_as(_u32p), len(offsets) - 1)

    def plain_encode(self, values):
        v = np.ascontiguousarray(values, dtype=np.float32).ravel()
        return self._new(self.lib.crcnn_plain_encode, "plain", v.ctypes.data_as(_f32p), len(v))

    def plain_encode_f64(self, values):
        """FractionalEncoder::encode on doubles (avg-pool's 1./(xf*yf), avgPoolingLayer.cpp:10-13)."""
        v = np.ascontiguousarray(values, dtype=np.float64).ravel()
        return self._new(self.lib.crcnn_plain_encode_f64, "plain", v.ctypes.data_as(C.POINTER(C.c_double)), len(v))

    def plain_get(self, p, index):
        out = np.zeros(self.stride, dtype=np.uint64)
        self._chk(self.lib.crcnn_plain_get(self.h, p.ptr, index, out.ctypes.data_as(_u64p)))
        return out

    def plain_get_ntt(self, p, index):
        out = np.zeros((self.K, self.stride), dtype=np.uint64)
        self._chk(self.lib.crcnn_plain_get_ntt(self.h, p.ptr, index, out.ctypes.data_as(_u64p)))
        return out

    def evk_upload(self, words, sizes, dbc=16):
        a = np.ascontiguousarray(words, dtype=np.uint64)
        s = np.ascontiguousarray(sizes, dtype=np.int32)
        return self._new(self.lib.crcnn_evk_upload, "evk", a.ctypes.data_as(_u64p), dbc, s.ctypes.data_as(_i32p))

    # ---- re-encryption on the device (opt-in: the key holder's keys next to the activations)
    def keys_upload(self, secret_key_ntt, public_key_ntt):
        sk = np.ascontiguousarray(secret_key_ntt, dtype=np.uint64)
        pk = np.ascontiguousarray(public_key_ntt, dtype=np.uint64)
        assert sk.size == self.K * self.stride and pk.size == 2 * self.K * self.stride
        return self._new(self.lib.crcnn_keys_upload, "keys", sk.ctypes.data, pk.ctypes.data)

    def decrypt(self, keys, t):
        """Decryptor::decrypt of every ciphertext of t -> [count][n+1] plaintext words."""
        out = np.zeros((self.count(t), self.stride), dtype=np.uint64)
        self._chk(self.lib.crcnn_decrypt(self.h, keys.ptr, t.ptr, out.ctypes.data))
        return out

    def noise_budget(self, keys, t):
        """Decryptor::invariant_noise_budget of every ciphertext of t -> int32[count]."""
        out = np.zeros(self.count(t), dtype=np.int32)
        self._chk(self.lib.crcnn_noise_budget(self.h, keys.ptr if keys is not None else None, t.ptr if t is not None else None,
                                              out.ctypes.data_as(_i32p), None))
        return out

    def min_noise_budget(self, keys, t):
        """The minimum invariant noise budget over t (crcnn_noise_budget's min_budget)."""
        m = C.c_int()
        self._chk(self.lib.crcnn_noise_budget(self.h, keys.ptr if keys is not None else None, t.ptr, None, C.byref(m)))
        return m.value

    def reencrypt(self, keys, t, seed=0, sigma=0.0, noise=None, want_plain=False):
        """decrypt -> decode -> float -> encode -> encrypt on the device; noise: optional int8 [count][3][n] (u, e0, e1).
        Returns the fresh tensor (and, with want_plain, the re-encoded plaintexts [count][n+1] and the decoded float values)."""
        cnt = self.count(t)
        nz = None
        if noise is not None:
            nz = np.ascontiguousarray(noise, dtype=np.int8)
            assert nz.size == cnt * 3 * self.n
        plain = np.zeros((cnt, self.stride), dtype=np.uint64) if want_plain else None
        vals = np.zeros(cnt, dtype=np.float32) if want_plain else None
        out = C.c_void_p()
        self._chk(self.lib.crcnn_reencrypt(self.h, keys.ptr, t.ptr, C.c_uint64(seed), C.c_double(sigma),
                                           nz.ctypes.data if nz is not None else None, C.byref(out),
                                           plain.ctypes.data if want_plain else None, vals.ctypes.data if want_plain else None))
        h = Handle(self, out, "tensor")
        return (h, plain, vals) if want_plain else h

    def encrypt_values(self, keys, values, seed=0, sigma=0.0, noise=None):
        """FractionalEncoder::encode + Encryptor::encrypt of every value (float32) on the device -> coefficient-form tensor of
        len(values) ciphertexts.  noise: optional int8 [count][3][n] (u, e0, e1) instead of the generator keyed by `seed`."""
        v = np.ascontiguousarray(values, dtype=np.float32).ravel()
        nz = None
        if noise is not None:
            nz = np.ascontiguousarray(noise, dtype=np.int8)
            assert nz.size == len(v) * 3 * self.n
        return self._new(self.lib.crcnn_encrypt_values, "tensor", keys.ptr if keys is not None else None, v.ctypes.data_as(_f32p), len(v),
                         C.c_uint64(seed), C.c_double(sigma), nz.ctypes.data if nz is not None else None)

    def decrypt_values(self, keys, t):
        """(float) FractionalEncoder::decode(Decryptor::decrypt(ct)) of every ciphertext of t -> float32[count]."""
        out = np.zeros(self.count(t), dtype=np.float32)
        self._chk(self.lib.crcnn_decrypt_values(self.h, keys.ptr if keys is not None else None, t.ptr, out.ctypes.data_as(_f32p)))
        return out

    # ---- layers
    def conv(self, x, w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, shard=None):
        if shard is None:
            return self._new(self.lib.crcnn_conv_forward, "tensor", x.ptr, w.ptr, b.ptr, batch, xd, yd, zd, xs, ys, xf, yf, nf)
        return self._new(self.lib.crcnn_conv_forward_shard, "tensor", x.ptr, w.ptr, b.ptr, batch, xd, yd, zd, xs, ys,
                         xf, yf, nf, shard[0], shard[1])

    def fc(self, x, w, b, batch, in_dim, out_dim, shard=None):
        if shard is None:
            return self._new(self.lib.crcnn_fc_forward, "tensor", x.ptr, w.ptr, b.ptr, batch, in_dim, out_dim)
        return self._new(self.lib.crcnn_fc_forward_shard, "tensor", x.ptr, w.ptr, b.ptr, batch, in_dim, out_dim,
                         shard[0], shard[1])

    def pool(self, x, batch, xd, yd, zd, xs, ys, xf, yf, scale=None):
        return self._new(self.lib.crcnn_pool_forward, "tensor", x.ptr, batch, xd, yd, zd, xs, ys, xf, yf,
                         scale.ptr if scale is not None else None)

    def bn(self, x, batch, zd, xd, yd, mean, invstd):
        return self._new(self.lib.crcnn_bn_forward, "tensor", x.ptr, batch, zd, xd, yd, mean.ptr, invstd.ptr)

    def conv_pool_bn(self, x, w, b, batch, xd, yd, zd, xs, ys, xf, yf, nf, pxs, pys, pxf, pyf, scale, mean, invstd, shard=None):
        """Convolution + average pooling + batch-norm on the pooled grid (crcnn_conv_pool_bn_forward[_shard])."""
        if shard is not None:
            return self._new(self.lib.crcnn_conv_pool_bn_forward_shard, "tensor", x.ptr, w.ptr, b.ptr, batch, xd, yd, zd, xs, ys, xf, yf, nf,
                             pxs, pys, pxf, pyf, scale.ptr if scale is not None else None, mean.ptr, invstd.ptr, shard[0], shard[1])
        return self._new(self.lib.crcnn_conv_pool_bn_forward, "tensor", x.ptr, w.ptr, b.ptr, batch, xd, yd, zd, xs, ys, xf, yf, nf,
                         pxs, pys, pxf, pyf, scale.ptr if scale is not None else None, mean.ptr, invstd.ptr)

    def pool_bn_fc_fc(self, x, batch, xd, yd, zd, pxs, pys, pxf, pyf, scale, mean, invstd, w1, b1, w2, b2, mid_dim, out_dim):
        """avg-pool + batch-norm + two fully connected layers as window sums + one composed layer (crcnn_pool_bn_fc_fc_forward)."""
        return self._new(self.lib.crcnn_pool_bn_fc_fc_forward, "tensor", x.ptr, batch, xd, yd, zd, pxs, pys, pxf, pyf, scale.ptr if scale is not None else None, mean.ptr,
                         invstd.ptr, w1.ptr, b1.ptr, w2.ptr, b2.ptr, mid_dim, out_dim)

    def fc_fc(self, x, w1, b1, w2, b2, batch, in_dim, mid_dim, out_dim):
        """Two fully connected layers in a row as one composed layer (crcnn_fc_fc_forward)."""
        return self._new(self.lib.crcnn_fc_fc_forward, "tensor", x.ptr, w1.ptr, b1.ptr, w2.ptr, b2.ptr, batch, in_dim, mid_dim, out_dim)

    def alloc_stats(self):
        """Allocator counters (crcnn_ctx_alloc_stats): dict of pool_mallocs, cache_hits, cache_bypass, flushes, small_mallocs, cached_bytes."""
        v = (C.c_longlong * 6)()
        self._chk(self.lib.crcnn_ctx_alloc_stats(self.h, v))
        return dict(zip(("pool_mallocs", "cache_hits", "cache_bypass", "flushes", "small_mallocs", "cached_bytes"), list(v)))

    def pool_bn(self, x, batch, xd, yd, zd, xs, ys, xf, yf, scale, mean, invstd):
        """Average pooling + batch-norm in one pass (crcnn_pool_bn_forward)."""
        return self._new(self.lib.crcnn_pool_bn_forward, "tensor", x.ptr, batch, xd, yd, zd, xs, ys, xf, yf, scale.ptr if scale is not None else None, mean.ptr, invstd.ptr)

    def square_layer(self, x, evk):
        return self._new(self.lib.crcnn_square_forward, "tensor", x.ptr, evk.ptr)

    # ---- evaluator-level
    def to_ntt(self, t):
        self._chk(self.lib.crcnn_transform_to_ntt(self.h, t.ptr))

    def from_ntt(self, t):
        self._chk(self.lib.crcnn_transform_from_ntt(self.h, t.ptr))

    def plain_op(self, t, p, index, op):
        self._chk(self.lib.crcnn_plain_op(self.h, t.ptr, p.ptr, index, {"mul": 0, "add": 1, "sub": 2}[op]))

    def add_many(self, t):
        return self._new(self.lib.crcnn_add_many, "tensor", t.ptr)

    def square(self, t):
        return self._new(self.lib.crcnn_square, "tensor", t.ptr)

    def relinearize(self, t3, evk):
        return self._new(self.lib.crcnn_relinearize, "tensor", t3.ptr, evk.ptr)

    # ---- measurement
    def prof_enable(self, on=True):
        self._chk(self.lib.crcnn_prof_enable(self.h, int(on)))

    def prof_reset(self):
        self._chk(self.lib.crcnn_prof_reset(self.h))

    def prof(self):
        out = {}
        name = C.create_string_buffer(32)
        for i in range(self.lib.crcnn_prof_count(self.h)):
            n, ms = C.c_long(), C.c_double()
            self._chk(self.lib.crcnn_prof_get(self.h, i, name, C.byref(n), C.byref(ms)))
            out[name.value.decode()] = (n.value, ms.value)
        return out

    def prof_work(self):
        """{class: (algorithmic bytes, algorithmic ops)} since the last reset (crcnn_prof_get_work)."""
        out = {}
        name = C.create_string_buffer(32)
        for i in range(self.lib.crcnn_prof_count(self.h)):
            n, ms, b, o = C.c_long(), C.c_double(), C.c_double(), C.c_double()
            self._chk(self.lib.crcnn_prof_get(self.h, i, name, C.byref(n), C.byref(ms)))
            self._chk(self.lib.crcnn_prof_get_work(self.h, i, C.byref(b), C.byref(o)))
            out[name.value.decode()] = (b.value, o.value)
        return out

    def probe_pipe(self, which, blocks, threads, iters):
        """(ops per second, ms) of roofline probe `which` (0: 64x64->128 MAC chain, 1: IMAD.WIDE issue rate, 2: UMMA kind::i8)."""
        ms, ops = C.c_double(), C.c_double()
        self._chk(self.lib.crcnn_probe_pipe(self.h, which, blocks, threads, iters, C.byref(ms), C.byref(ops)))
        return ops.value / (ms.value / 1000.0), ms.value

    def probe_imad(self, blocks, threads, iters):
        ms = C.c_double()
        self._chk(self.lib.crcnn_probe_imad(self.h, blocks, threads, iters, C.byref(ms)))
        return ms.value
