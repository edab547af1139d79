"""ctypes plumbing over crcnn_b200/libcrcnn_b200_host.so: the C++17 host path (crcnn_b200/cpp/: Runtime, CnnBuilder, Network,
ShardedNetwork, BatchServer) that a CrCNN program links, driven from the harness.  bench.py measures through this, so the
headline numbers come from the C++ predict path and serving loop, not from Python glue.  One network per process."""
import ctypes as C
import os
import tempfile

import numpy as np

from . import lib as _lib
from . import nets
from .h5write import write_h5

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_HERE, "libcrcnn_b200_host.so")
TOPOLOGY_OF = {"PlainModel": "PlainModel", "ApproxPlainModel": "Approx", "PlainModelWoPad": "WoPad", "PlainModelTiny": "Tiny"}
_vp, _I, _dp = C.c_void_p, C.c_int, C.POINTER(C.c_double)

_h = None


def load():
    global _h
    if _h is not None:
        return _h
    _lib.load()
    if not os.path.exists(HOST_LIB_PATH):
        raise RuntimeError("crcnn_b200/libcrcnn_b200_host.so is missing: build it with `make -C crcnn_b200/csrc`")
    h = C.CDLL(HOST_LIB_PATH)
    h.crcnn_host_last_error.restype = C.c_char_p
    h.crcnn_host_ctx.restype = _vp
    h.crcnn_host_init.argtypes = [_I, _I, _vp, C.c_uint64, _I]
    h.crcnn_host_set_evk.argtypes = [_vp, _vp, _I]
    h.crcnn_host_build.argtypes = [C.c_char_p, C.c_char_p, _I, _I, _vp, _I]
    h.crcnn_host_shape.argtypes = [C.POINTER(_I)] * 5
    h.crcnn_host_layer_name.argtypes = [_I, C.c_char_p, _I]
    h.crcnn_host_forward_range.argtypes = [_vp, _I, _I, _I, _I, _I, _I, _vp, C.c_long, C.POINTER(_I)]
    h.crcnn_host_resident_begin.argtypes = [_vp, _I]
    h.crcnn_host_resident_run.argtypes = [_I, _dp, _dp, _vp]
    h.crcnn_host_serve.argtypes = [_vp, _vp, _I, C.c_long, _dp]
    h.crcnn_host_set_fusion.argtypes = [_I]
    h.crcnn_host_serve_times.argtypes = [_dp, _I]
    h.crcnn_host_serve_times.restype = _I
    h.crcnn_host_use_keys.argtypes = [_vp, _vp, _I, C.c_uint64]
    h.crcnn_host_set_budget_threshold.argtypes = [_I]
    h.crcnn_host_forward_adaptive.argtypes = [_vp, _I, _vp, C.c_long, C.POINTER(_I), C.POINTER(_I)]
    h.crcnn_host_budget_log.argtypes = [C.POINTER(_I)] * 3 + [_I]
    h.crcnn_host_budget_log.restype = _I
    h.crcnn_host_predict_values.argtypes = [C.POINTER(C.c_float), _I, C.c_uint64, C.POINTER(C.c_float), C.POINTER(_I)]
    _h = h
    return h


class HostError(RuntimeError):
    pass


CRCNN_ERR_OUT_OF_BUDGET = -6


class OutOfBudget(HostError):
    """OutOfBudgetException of the host library: the activation after `layer` has no noise budget left to go on with."""

    def __init__(self, msg, layer):
        super().__init__(msg)
        self.layer = layer


def weights_h5(model, directory=None):
    """The model's trained tensors as an .h5 file CnnBuilder can read (the reference's PlainModel*.h5 are not on the GPU box;
    weights/*.npz hold the same float32 tensors, tools/export_weights.py)."""
    directory = directory or tempfile.gettempdir()
    path = os.path.join(directory, "crcnn_b200_%s_%d.h5" % (model, os.getpid()))
    write_h5(path, nets.load_weights(model))
    return path


class HostNetwork:
    """Runtime::init + CnnBuilder(h5).buildNetwork(topology) [+ ShardedNetwork over NCCL] in the C++ host library."""

    def __init__(self, n, primes, t, model, device=0, evk=None, world=1, rank=0, nccl_id=None, skip_reencryption=True, h5_path=None):
        self.h = load()
        self.n, self.K, self.t = int(n), len(primes), int(t)
        self.stride = self.n + 1
        q = np.array([int(p) for p in primes], dtype=np.uint64)
        self._chk(self.h.crcnn_host_init(self.n, self.K, q.ctypes.data, self.t, device))
        if evk is not None:
            words, sizes, dbc = evk
            w = np.ascontiguousarray(words, dtype=np.uint64)
            s = np.ascontiguousarray(sizes, dtype=np.int32)
            self._chk(self.h.crcnn_host_set_evk(w.ctypes.data, s.ctypes.data, int(dbc)))
        own = h5_path is None
        path = h5_path or weights_h5(model)
        try:
            idbuf = (C.c_char * 128).from_buffer_copy(nccl_id) if nccl_id is not None else None
            self._chk(self.h.crcnn_host_build(path.encode(), TOPOLOGY_OF.get(model, model).encode(), world, rank,
                                              C.cast(idbuf, _vp) if idbuf is not None else None, int(skip_reencryption)))
        finally:
            if own:
                os.unlink(path)
        v = [_I() for _ in range(5)]
        self._chk(self.h.crcnn_host_shape(*[C.byref(x) for x in v]))
        self.zd, self.xd, self.yd, self.outputs, self.num_layers = [x.value for x in v]
        name = C.create_string_buffer(128)
        self.layer_names = []
        for i in range(self.num_layers):
            self.h.crcnn_host_layer_name(i, name, 128)
            self.layer_names.append(name.value.decode())

    def _chk(self, rc):
        if rc != 0:
            raise HostError("crcnn_b200 host error %d: %s" % (rc, self.h.crcnn_host_last_error().decode()))

    def ctx(self):
        """The crcnn_ctx* of the C++ Runtime (for the profiling / probe entry points of the C ABI)."""
        return self.h.crcnn_host_ctx()

    def ct_words(self):
        return 2 * self.K * self.stride

    def forward(self, x, batch=1, first=0, last=None, shape=None):
        """Layers [first,last) on host ciphertexts x ([batch * z*x*y][2][K][n+1]); returns (output array, (z, x, y))."""
        x = np.ascontiguousarray(x, dtype=np.uint64)
        zd, xd, yd = shape or (self.zd, self.xd, self.yd)
        last = self.num_layers if last is None else last
        cap = max(x.size, batch * 64 * 64 * 64 * 2 * self.K * self.stride // 64)
        out = np.empty(cap, dtype=np.uint64)
        oshape = (_I * 3)()
        self._chk(self.h.crcnn_host_forward_range(x.ctypes.data, batch, zd, xd, yd, first, last, out.ctypes.data, cap, oshape))
        z, a, b = oshape[0], oshape[1], oshape[2]
        cnt = batch * z * a * b
        return out[:cnt * self.ct_words()].reshape(cnt, 2, self.K, self.stride).copy(), (z, a, b)

    def resident_begin(self, pinned_ptr, batch):
        """Upload the batch once; resident_run() then times forwards that start from a fresh device copy of it."""
        self._chk(self.h.crcnn_host_resident_begin(pinned_ptr, batch))
        self.resident_batch = batch

    def resident_run(self, steps, out=None):
        """(total ms by CUDA events, [ms per layer]) of `steps` forwards of the resident batch.  out: a uint64 array of
        [batch * outputs][2][K][n+1] words that receives the scores of the last of those forwards."""
        ms = C.c_double()
        per = (C.c_double * self.num_layers)()
        if out is not None and not (out.dtype == np.uint64 and out.flags.c_contiguous and out.flags.writeable
                                    and out.size == self.resident_batch * self.outputs * self.ct_words()):
            raise ValueError("out must be a writable contiguous uint64 array of batch * outputs ciphertexts")
        self._chk(self.h.crcnn_host_resident_run(steps, C.byref(ms), per, None if out is None else out.ctypes.data))
        return ms.value, list(per)

    def resident_end(self):
        self._chk(self.h.crcnn_host_resident_end())

    def resident_steps(self, pinned_ptr, batch, warmup, steps):
        self.resident_begin(pinned_ptr, batch)
        if warmup:
            self.resident_run(warmup)
        out = self.resident_run(steps)
        self.resident_end()
        return out

    def serve(self, pinned_in_ptr, pinned_out_ptr, batch, requests):
        ms = C.c_double()
        self._chk(self.h.crcnn_host_serve(pinned_in_ptr, pinned_out_ptr, batch, requests, C.byref(ms)))
        return ms.value

    def use_keys(self, secret_key_ntt, public_key_ntt, device_reencryption=False, seed=0):
        """Network::use_device_keys (or use_device_reencryption with `seed`): the key holder's keys on the device."""
        sk = np.ascontiguousarray(secret_key_ntt, dtype=np.uint64)
        pk = np.ascontiguousarray(public_key_ntt, dtype=np.uint64)
        assert sk.size == self.K * self.stride and pk.size == 2 * self.K * self.stride
        self._chk(self.h.crcnn_host_use_keys(sk.ctypes.data, pk.ctypes.data, int(bool(device_reencryption)), C.c_uint64(seed)))

    def set_budget_threshold(self, threshold):
        """Network::reencrypt_below_budget: -1 keeps the fixed re-encryption point, >= 0 re-encrypts when the budget falls to it."""
        self._chk(self.h.crcnn_host_set_budget_threshold(int(threshold)))

    def forward_adaptive(self, x, batch=1):
        """Network::forward_dev_adaptive on host ciphertexts x ([batch * z*x*y][2][K][n+1]) -> (output array, (z, x, y)).
        Raises OutOfBudget (with .layer) where the network throws OutOfBudgetException."""
        x = np.ascontiguousarray(x, dtype=np.uint64)
        cap = max(x.size, batch * 64 * 64 * 64 * 2 * self.K * self.stride // 64)
        out = np.empty(cap, dtype=np.uint64)
        oshape, failed = (_I * 3)(), _I(-1)
        rc = self.h.crcnn_host_forward_adaptive(x.ctypes.data, batch, out.ctypes.data, cap, oshape, C.byref(failed))
        if rc == CRCNN_ERR_OUT_OF_BUDGET:
            raise OutOfBudget(self.h.crcnn_host_last_error().decode(), failed.value)
        self._chk(rc)
        cnt = batch * oshape[0] * oshape[1] * oshape[2]
        return out[:cnt * self.ct_words()].reshape(cnt, 2, self.K, self.stride).copy(), (oshape[0], oshape[1], oshape[2])

    def predict_values(self, images, batch=1, seed=0):
        """Network::predict: float32 images ([batch][z][x][y] values) encrypted on the device with the keys of use_keys, the network's
        forward (as forward_batch runs it), the scores decrypted on the device -> float32 [batch][outputs].  Each call draws its
        randomness from (seed, call number).  Raises OutOfBudget (with .layer) where the network throws OutOfBudgetException."""
        x = np.ascontiguousarray(images, dtype=np.float32).ravel()
        if x.size != batch * self.zd * self.xd * self.yd:
            raise ValueError("images must hold batch * %d values" % (self.zd * self.xd * self.yd))
        out = np.zeros((batch, self.outputs), dtype=np.float32)
        fp = C.POINTER(C.c_float)
        failed = _I(-1)
        rc = self.h.crcnn_host_predict_values(x.ctypes.data_as(fp), batch, C.c_uint64(seed), out.ctypes.data_as(fp), C.byref(failed))
        if rc == CRCNN_ERR_OUT_OF_BUDGET:
            raise OutOfBudget(self.h.crcnn_host_last_error().decode(), failed.value)
        self._chk(rc)
        return out

    def budget_log(self):
        """Network::budget_log of the last adaptive forward: [(layer, min budget, re-encrypted)]."""
        cap = 256
        a, b, c = (_I * cap)(), (_I * cap)(), (_I * cap)()
        k = min(self.h.crcnn_host_budget_log(a, b, c, cap), cap)
        return [(a[i], b[i], bool(c[i])) for i in range(k)]

    def set_fusion(self, on):
        """Layer fusion (conv+pool+bn on the pooled grid, pool+bn, fc+fc composed) on / off; off = one call per reference layer."""
        self._chk(self.h.crcnn_host_set_fusion(int(bool(on))))

    def serve_times(self):
        """ms (host clock, from the start of the last serve()) at which each request's scores had landed."""
        buf = (C.c_double * 4096)()
        k = self.h.crcnn_host_serve_times(buf, 4096)
        return list(buf[:min(k, 4096)])

    def close(self):
        self.h.crcnn_host_shutdown()


def pinned_array(words):
    """numpy uint64 view of `words` words of page-locked host memory (crcnn_pinned_alloc); keep the returned owner alive."""
    L = _lib.load()
    p = C.c_void_p()
    if L.crcnn_pinned_alloc(C.c_size_t(words * 8), C.byref(p)) != 0:
        raise MemoryError("crcnn_pinned_alloc(%d bytes) failed" % (words * 8))
    buf = (C.c_uint64 * words).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.uint64)

    class _Owner:
        ptr = p.value

        def __del__(self):
            try:
                L.crcnn_pinned_free(C.c_void_p(self.ptr))
            except Exception:
                pass
    return arr, _Owner()


def nccl_unique_id():
    L = _lib.load()
    buf = C.create_string_buffer(128)
    rc = L.crcnn_comm_unique_id(buf)
    if rc != 0:
        raise HostError("crcnn_comm_unique_id failed: %s" % L.crcnn_last_error(None).decode())
    return buf.raw
