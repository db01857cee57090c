"""
FITC sparse pseudo-input GP on the device (pygp/inference/fitc.py:19-232).

Same constructor, properties and error behaviour as the reference; `_update`,
`loglikelihood` and `_marg_posterior(grad=False)` are single C-ABI calls
(pgp_fitc_update / _loglike / _predict).  X, y, U and every (n, p) intermediate
stay in HBM; only the hyper vector goes in and (lZ, dlZ) / (mu, s2) come out.

Beyond the reference: the pseudo-inputs can be moved (`set_pseudoinputs`) and
`loglikelihood(grad=True, pseudoinputs=True)` also returns d lZ / d U, so that
`learning.optimize(gp, pseudoinputs=True)` can fit the inducing set.
"""

import ctypes as C

import numpy as np

from .. import _lib
from ..likelihoods import Gaussian
from ._base import GP

__all__ = ['FITC']


class _DeviceFITC(object):
    """Owner of a `pgp_fitc*`.  A deep copy (Parameterized.copy) starts without
    device state; the copy rebuilds its own lazily (`FITC._ensure_dev`) the first
    time it is evaluated, so `gp.copy().posterior(X)` works as in the reference."""

    def __init__(self, ctx, handle):
        self.ctx, self.handle = ctx, handle

    @classmethod
    def create(cls, kernel, U, X, y, dtc=False):
        ctx = _lib.context()
        U, X, y = _lib.as_f64(U, 2), _lib.as_f64(X, 2), _lib.as_f64(y, 1)
        h = C.c_void_p()
        make = _lib.lib().pgp_dtc_create if dtc else _lib.lib().pgp_fitc_create
        _lib.check(ctx, make(ctx.handle, kernel._spec(), _lib.ptr(U), len(U), _lib.ptr(X), _lib.ptr(y), len(X),
                             C.byref(h)))
        return cls(ctx, h)

    def __deepcopy__(self, memo):
        return None

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().pgp_fitc_destroy(self.handle)
                self.handle = None
        except Exception:       # interpreter shutdown
            pass


class FITC(GP):
    """GP inference using sparse pseudo-inputs."""

    _dtc = False        # DTC (inference/dtc.py) runs the same device state with the dtc.py algebra

    def __init__(self, likelihood, kernel, mean, U):
        # exact FITC inference only works with Gaussian likelihoods (fitc.py:24-26)
        if not isinstance(likelihood, Gaussian):
            raise ValueError('exact inference requires a Gaussian likelihood')
        super(FITC, self).__init__(likelihood, kernel, mean)
        self._U = np.array(U, ndmin=2, dtype=float, copy=True)
        if self._U.shape[1] != self._kernel.ndim:
            raise ValueError('pseudo-inputs have the wrong number of columns')
        self._dev = None
        self._ndev = 0

    def reset(self):
        self._dev = None
        self._ndev = 0
        super(FITC, self).reset()

    @property
    def pseudoinputs(self):
        """The pseudo-input points."""
        return self._U

    def set_pseudoinputs(self, U):
        """Move the pseudo-inputs to the rows of U (a copy is kept) and, if data
        is present, re-factorise, as `set_hyper` does.  U may have a different
        number of rows; its columns must match the kernel's inputs."""
        self._set_pseudoinputs(U)
        if self.ndata > 0:
            self._update()

    def _set_pseudoinputs(self, U):
        """Replace U without re-factorising: the device state stays unfactored
        until the next `_update` (set_hyper / add_data)."""
        U = np.array(U, ndmin=2, dtype=float, copy=True)
        if U.shape[1] != self._kernel.ndim:
            raise ValueError('pseudo-inputs have the wrong number of columns')
        if self._dev is not None and U.shape[0] == self._U.shape[0]:
            _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_set_pseudoinputs(self._dev.handle, _lib.ptr(U)))
        else:
            self._dev = None            # a different p: rebuilt by the next _update
            self._ndev = 0
        self._U = U

    @classmethod
    def from_gp(cls, gp, U=None):
        if U is None:
            if hasattr(gp, 'pseudoinputs'):
                U = gp.pseudoinputs.copy()
            else:
                raise ValueError('gp has no pseudoinputs and none are given')
        newgp = cls(gp._likelihood.copy(), gp._kernel.copy(), gp._mean, U)
        if gp.ndata > 0:
            X, y = gp.data
            newgp.add_data(X, y)
        return newgp

    def _update(self):
        if self._dev is None or self._ndev != self.ndata:
            # new rows that did not go through _updateinc (the reference refactors
            # on every add_data, _base.py:133-141): upload all the data again
            self._dev = None
            self._dev = _DeviceFITC.create(self._kernel, self._U, self._X, self._y, self._dtc)
            self._ndev = self.ndata
        hyp = _lib.as_f64(self.get_hyper())
        _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_update(self._dev.handle, _lib.ptr(hyp)))

    def _updateinc(self, X, y):
        """Append rows to a factored device state by rank updates of its p x p
        factors, O(len(X) p^2) whatever ndata is (pgp_fitc_append_inc; beyond the
        reference, which refactors on all the data).  At most min(ndata, the
        library's row cap) rows: past ndata new rows the full update costs less
        than twice the incremental one, and it is the reference path."""
        dev = self._dev
        if dev is None or self._ndev != self.ndata or len(X) > self.ndata:
            raise NotImplementedError
        if len(X) > _lib.lib().pgp_fitc_inc_max_rows():
            raise NotImplementedError
        Xn, yn = _lib.as_f64(X, 2), _lib.as_f64(y, 1)
        rc = _lib.lib().pgp_fitc_append_inc(dev.handle, _lib.ptr(Xn), _lib.ptr(yn), len(Xn))
        if rc == -4:
            raise NotImplementedError       # not factored (set_pseudoinputs): the full update takes over
        try:
            _lib.check(dev.ctx, rc)
        except Exception:
            # the handle is unfactored now: drop it, the next _update uploads the host's data again
            self._dev, self._ndev = None, 0
            raise
        self._ndev += len(Xn)

    def _ensure_dev(self):
        """Device state of a copy made without a hyper argument (utils/models.py:47-55):
        rebuilt on first use from the host data the copy carries."""
        if self._dev is None and self.ndata > 0:
            self._update()

    def loglikelihood(self, grad=False, pseudoinputs=False):
        """lZ; with `grad`, (lZ, dlZ); with `pseudoinputs`, (lZ, dlZ, dU), where
        dU = d lZ / d U has the shape of `pseudoinputs` (lZ and dlZ are bitwise
        those of `loglikelihood(True)`)."""
        self._ensure_dev()
        lZ = C.c_double()
        if pseudoinputs:
            dlZ, dU = np.empty(self.nhyper), np.empty(self._U.shape)
            _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_loglike_pseudo(
                self._dev.handle, C.byref(lZ), _lib.ptr(dlZ), _lib.ptr(dU)))
            return lZ.value, dlZ, dU
        dlZ = np.empty(self.nhyper) if grad else None
        _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_loglike(
            self._dev.handle, int(bool(grad)), C.byref(lZ), None if dlZ is None else _lib.ptr(dlZ)))
        return (lZ.value, dlZ) if grad else lZ.value

    def _full_posterior(self, X):
        """Joint posterior mean and covariance at the rows of X (fitc.py:102-120)."""
        X = _lib.as_f64(X, 2)
        if self._X is None:
            return np.full(X.shape[0], self._mean), self._kernel.get(X)
        self._ensure_dev()
        mu, Sigma = np.empty(len(X)), np.empty((len(X), len(X)))
        _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_full_posterior(
            self._dev.handle, _lib.ptr(X), len(X), _lib.ptr(mu), _lib.ptr(Sigma)))
        return mu, Sigma

    def _marg_posterior(self, X, grad=False):
        X = _lib.as_f64(X, 2)
        if self._X is None:
            out = (np.full(X.shape[0], self._mean), self._kernel.dget(X))
            return out + (np.zeros_like(X), np.zeros_like(X)) if grad else out
        if X.shape[1] != self._kernel.ndim:
            raise ValueError('test inputs have the wrong number of columns')
        self._ensure_dev()
        mu, s2 = np.empty(len(X)), np.empty(len(X))
        if not grad:
            _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_predict(
                self._dev.handle, _lib.ptr(X), len(X), _lib.ptr(mu), _lib.ptr(s2)))
            return mu, s2
        dmu, ds2 = np.empty(X.shape), np.empty(X.shape)
        _lib.check(self._dev.ctx, _lib.lib().pgp_fitc_predict_grad(
            self._dev.handle, _lib.ptr(X), len(X), _lib.ptr(mu), _lib.ptr(s2), _lib.ptr(dmu), _lib.ptr(ds2)))
        return mu, s2, dmu, ds2
