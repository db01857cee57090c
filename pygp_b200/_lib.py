"""
ctypes binding of libpygp_b200.so (include/pygp_b200.h).

This is the ONLY arithmetic path of the package: there is no numpy/CPU
fallback.  If the shared library or a CUDA device is missing every operation
raises (`LibraryNotBuilt` / `RuntimeError`) instead of degrading.
"""

import ctypes as C
import os
import threading

import numpy as np

__all__ = ['lib', 'context', 'KernelSpec', 'check', 'LibraryNotBuilt',
           'MAX_PARTS', 'MAX_OPS', 'MAX_DIM', 'MAX_HYPER', 'as_f64', 'ptr']

MAX_PARTS, MAX_OPS, MAX_DIM, MAX_HYPER = 8, 16, 64, 96
SE, MATERN1, MATERN3, MATERN5, PERIODIC, RQ = range(6)
OP_PUSH, OP_SUM, OP_PROD = range(3)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libpygp_b200.so')


class LibraryNotBuilt(ImportError):
    pass


class Part(C.Structure):
    _fields_ = [('type', C.c_int32), ('iso', C.c_int32),
                ('hyper_offset', C.c_int32), ('nhyper', C.c_int32)]


class Op(C.Structure):
    _fields_ = [('op', C.c_int32), ('arg', C.c_int32)]


class KernelSpec(C.Structure):
    _fields_ = [('ndim', C.c_int32), ('nhyper', C.c_int32),
                ('n_parts', C.c_int32), ('n_ops', C.c_int32),
                ('parts', Part * MAX_PARTS), ('ops', Op * MAX_OPS)]


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_vp = C.c_void_p
_i64 = C.c_int64
_sp = C.POINTER(KernelSpec)

# name -> (restype, argtypes): every symbol include/pygp_b200.h declares
SIGNATURES = {
    'pgp_abi_version': (C.c_int, []),
    'pgp_ctx_create': (C.c_int, [C.c_int, C.POINTER(_vp)]),
    'pgp_ctx_destroy': (None, [_vp]),
    'pgp_last_error': (C.c_char_p, [_vp]),
    'pgp_ctx_stream': (_vp, [_vp]),
    'pgp_ctx_sync': (C.c_int, [_vp]),
    'pgp_ctx_launch_count': (_i64, [_vp]),
    'pgp_ctx_profile': (C.c_int, [_vp, C.c_int]),
    'pgp_ctx_profile_read': (C.c_int, [_vp, C.c_int, C.POINTER(_i64), _dp, _dp]),
    'pgp_gram': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, _dp]),
    'pgp_gram_grad': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, C.c_int32, _dp]),
    'pgp_dget': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp]),
    'pgp_dgrad': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp]),
    'pgp_gram_gradx': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, C.c_int32, _dp]),
    'pgp_gram_gradxy': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, _dp]),
    'pgp_gram_dev': (C.c_int, [_vp, _sp, _dp, _vp, _i64, _vp, _i64, _vp]),
    'pgp_exact_create': (C.c_int, [_vp, _sp, _dp, _dp, _i64, C.POINTER(_vp)]),
    'pgp_exact_append': (C.c_int, [_vp, _dp, _dp, _i64]),
    'pgp_exact_append_inc': (C.c_int, [_vp, _dp, _dp, _i64]),
    'pgp_model_clone': (C.c_int, [_vp, C.POINTER(_vp)]),
    'pgp_model_destroy': (None, [_vp]),
    'pgp_model_ndata': (_i64, [_vp]),
    'pgp_exact_update': (C.c_int, [_vp, _dp]),
    'pgp_exact_loglike': (C.c_int, [_vp, C.c_int, _dp, _dp]),
    'pgp_exact_predict': (C.c_int, [_vp, _dp, _i64, _dp, _dp]),
    'pgp_exact_predict_grad': (C.c_int, [_vp, _dp, _i64, _dp, _dp, _dp, _dp]),
    'pgp_exact_predict_dev': (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    'pgp_exact_full_posterior': (C.c_int, [_vp, _dp, _i64, _dp, _dp]),
    'pgp_mvn_transform': (C.c_int, [_vp, _dp, _dp, _i64, C.c_double, _dp, _i64, _dp]),
    'pgp_exact_get_factor': (C.c_int, [_vp, _dp, _dp]),
    'pgp_exact_factor_buffer': (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_i64)]),
    'pgp_exact_adopt_factor': (C.c_int, [_vp, _dp]),
    'pgp_dist_unique_id': (C.c_int, [_vp, _vp]),
    'pgp_dist_init': (C.c_int, [_vp, C.c_int, C.c_int, _vp, C.POINTER(_vp)]),
    'pgp_dist_destroy': (None, [_vp]),
    'pgp_dist_rank': (C.c_int, [_vp]),
    'pgp_dist_size': (C.c_int, [_vp]),
    'pgp_dist_set_group': (C.c_int, [_vp, _i64]),
    'pgp_dist_set_chunks': (C.c_int, [_vp, C.c_int]),
    'pgp_dist_allreduce': (C.c_int, [_vp, _dp, _i64, C.c_int]),
    'pgp_dist_exact_update': (C.c_int, [_vp, _vp, _dp, _i64]),
    'pgp_dist_exact_loglike': (C.c_int, [_vp, _vp, _i64, C.c_int, _dp, _dp]),
    'pgp_batched_loglike': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, _dp, _dp, _ip]),
    'pgp_batched_predict': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, _dp, _i64, _dp, _dp, _ip]),
    'pgp_batch_create': (C.c_int, [_vp, _sp, _dp, _dp, _i64, _dp, _i64, _i64, C.POINTER(_vp), _ip]),
    'pgp_batch_predict': (C.c_int, [_vp, _dp, _i64, _dp, _dp, _dp, _dp]),
    'pgp_batch_resident': (_i64, [_vp]),
    'pgp_batch_destroy': (None, [_vp]),
    'pgp_fitc_create': (C.c_int, [_vp, _sp, _dp, _i64, _dp, _dp, _i64, C.POINTER(_vp)]),
    'pgp_dtc_create': (C.c_int, [_vp, _sp, _dp, _i64, _dp, _dp, _i64, C.POINTER(_vp)]),
    'pgp_fitc_destroy': (None, [_vp]),
    'pgp_fitc_update': (C.c_int, [_vp, _dp]),
    'pgp_fitc_append_inc': (C.c_int, [_vp, _dp, _dp, _i64]),
    'pgp_fitc_inc_max_rows': (C.c_int, []),
    'pgp_fitc_loglike': (C.c_int, [_vp, C.c_int, _dp, _dp]),
    'pgp_fitc_loglike_pseudo': (C.c_int, [_vp, _dp, _dp, _dp]),
    'pgp_fitc_set_pseudoinputs': (C.c_int, [_vp, _dp]),
    'pgp_fitc_predict': (C.c_int, [_vp, _dp, _i64, _dp, _dp]),
    'pgp_fitc_full_posterior': (C.c_int, [_vp, _dp, _i64, _dp, _dp]),
    'pgp_fitc_predict_grad': (C.c_int, [_vp, _dp, _i64, _dp, _dp, _dp, _dp]),
    'pgp_dev_gemm_nt': (C.c_int, [_vp, _i64, _i64, _i64, C.c_double, _vp, _i64, _vp, _i64,
                                  C.c_double, _vp, _i64, C.c_int]),
    'pgp_dev_gemm': (C.c_int, [_vp, C.c_int, C.c_int, _i64, _i64, _i64, C.c_double, _vp, _i64, _vp, _i64,
                               C.c_double, _vp, _i64, C.c_int, C.c_int]),
    'pgp_dev_trsm': (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, C.c_int]),
    'pgp_dev_copy2d': (C.c_int, [_vp, _vp, _i64, _vp, _i64, _i64, _i64]),
    'pgp_dev_potrf': (C.c_int, [_vp, _vp, _i64, _i64, _i64]),
    'pgp_dev_chol_update': (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _i64]),
    'pgp_dev_fastmath': (C.c_int, [_vp, C.c_int, _dp, _i64, _dp]),
}

_lib = None
_lock = threading.RLock()
_contexts = {}


def lib():
    """Load libpygp_b200.so (once) and declare every signature."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise LibraryNotBuilt(
                        '%s not found: build it with `python -c "import __graft_entry__ as g; '
                        'g.build()"` or `make -C pygp_b200/csrc` (there is no CPU fallback)'
                        % LIB_PATH)
                handle = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)      # AttributeError if the .so lacks it
                    fn.restype = res
                    fn.argtypes = args
                if handle.pgp_abi_version() != 2:
                    raise LibraryNotBuilt('libpygp_b200.so ABI version mismatch')
                _lib = handle
    return _lib


class Context(object):
    """One per (process, device): owns the CUDA stream all work runs on."""

    def __init__(self, device):
        self.device = device
        h = _vp()
        rc = lib().pgp_ctx_create(device, C.byref(h))
        if rc != 0:
            msg = lib().pgp_last_error(None).decode()
            raise RuntimeError('pgp_ctx_create(device=%d) failed: %s' % (device, msg))
        self.handle = h

    def last_error(self):
        return lib().pgp_last_error(self.handle).decode()

    def sync(self):
        check(self, lib().pgp_ctx_sync(self.handle))

    @property
    def stream(self):
        return lib().pgp_ctx_stream(self.handle)

    @property
    def launch_count(self):
        return int(lib().pgp_ctx_launch_count(self.handle))

    def profile(self, enable):
        check(self, lib().pgp_ctx_profile(self.handle, int(bool(enable))))

    def profile_read(self, cls):
        n, ms, work = _i64(), C.c_double(), C.c_double()
        check(self, lib().pgp_ctx_profile_read(self.handle, cls, C.byref(n), C.byref(ms), C.byref(work)))
        return int(n.value), float(ms.value), float(work.value)


def default_device():
    dev = os.environ.get('PYGP_B200_DEVICE')
    if dev is None:
        dev = os.environ.get('LOCAL_RANK', '0')      # one process per GPU under torchrun
    return int(dev)


def context(device=None):
    device = default_device() if device is None else int(device)
    lib()
    ctx = _contexts.get(device)
    if ctx is None:
        with _lock:
            ctx = _contexts.get(device)
            if ctx is None:
                ctx = _contexts[device] = Context(device)
    return ctx


def check(ctx, rc):
    """Map a C return code to the exception the reference would raise."""
    if rc == 0:
        return
    msg = ctx.last_error() if ctx is not None else lib().pgp_last_error(None).decode()
    if rc > 0:
        # scipy.linalg.cholesky failure in the reference (exact.py:54)
        raise np.linalg.LinAlgError(msg or '%d-th leading minor of the array is not positive definite' % rc)
    if rc == -1:
        raise ValueError(msg)
    if rc == -3:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def as_f64(a, ndmin=1):
    return np.ascontiguousarray(np.array(a, dtype=np.float64, ndmin=ndmin))


def ptr(a):
    return a.ctypes.data_as(_dp)
