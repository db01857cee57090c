"""
Hyper-parameter marginalisation by MCMC (pygp/meta/mcmc.py:22-93).

The reference keeps n deep copies of the GP (one factorisation each) and loops
over them in `posterior`.  Here, for an ExactGP, the n sampled hyper vectors
are one resident batch on the device (`pgp_batch`: the n factorisations done
once, by the same launches, and kept in HBM while the chain is unchanged), and
the mixture prediction -- with or without input-gradients -- is ONE batched
call on it.  Model objects are materialised only when iterated.
"""

import copy
import ctypes as C

import numpy as np

from .. import _lib
from ..inference.exact import ExactGP
from ..learning.sampling import sample
from ..utils.random import rstate

__all__ = ['MCMC']


class _DeviceBatch(object):
    """Owner of a `pgp_batch*`: the exact GPs of one data set under the rows of `hypers`, factored on
    creation.  `budget` bytes (0: half the free device memory) bound the factors kept resident; the
    others are factored again at every predict."""

    def __init__(self, model, hypers, budget=0):
        self.ctx, self.handle = _lib.context(), None
        X, y = _lib.as_f64(model._X, 2), _lib.as_f64(model._y, 1)
        H = _lib.as_f64(hypers, 2)
        self.B, self.ndim = len(H), model._kernel.ndim
        self.info = np.zeros(self.B, dtype=np.int32)
        h = C.c_void_p()
        _lib.check(self.ctx, _lib.lib().pgp_batch_create(
            self.ctx.handle, model._kernel._spec(), _lib.ptr(X), _lib.ptr(y), len(X), _lib.ptr(H), self.B,
            int(budget), C.byref(h), self.info.ctypes.data_as(C.POINTER(C.c_int32))))
        self.handle = h

    @property
    def resident(self):
        return int(_lib.lib().pgp_batch_resident(self.handle))

    def predict(self, X, grad=False):
        """Per-problem posteriors at the rows of X (already transformed): mu, s2 (B, m) and, with grad,
        dmu, ds2 (B, m, ndim)."""
        if np.any(self.info):
            raise np.linalg.LinAlgError('sampled hyper-parameters give a non positive definite kernel matrix')
        X = _lib.as_f64(X, 2)
        if X.shape[1] != self.ndim:
            raise ValueError('test inputs have the wrong number of columns')
        m = len(X)
        mu, s2 = np.empty((self.B, m)), np.empty((self.B, m))
        dmu = np.empty((self.B, m, self.ndim)) if grad else None
        ds2 = np.empty((self.B, m, self.ndim)) if grad else None
        _lib.check(self.ctx, _lib.lib().pgp_batch_predict(
            self.handle, _lib.ptr(X), m, _lib.ptr(mu), _lib.ptr(s2),
            None if dmu is None else _lib.ptr(dmu), None if ds2 is None else _lib.ptr(ds2)))
        return (mu, s2, dmu, ds2) if grad else (mu, s2)

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().pgp_batch_destroy(self.handle)
                self.handle = None
        except Exception:       # interpreter shutdown
            pass


def _mixture(mu_, s2_, dmu_=None, ds2_=None):
    """Moment-matched mixture of the components (mcmc.py:75-93)."""
    mu = np.mean(mu_, axis=0)
    s2 = np.mean(s2_ + (mu_ - mu)**2, axis=0)
    if dmu_ is None:
        return mu, s2
    dmu = np.mean(dmu_, axis=0)
    Dmu = dmu_ - dmu
    ds2 = np.mean(ds2_ + 2*mu_[:, :, None]*Dmu - 2*mu[None, :, None]*Dmu, axis=0)
    return mu, s2, dmu, ds2


class MCMC(object):
    # Opt-in multi-GPU mixture (SURVEY.md 8e): set `sharded = True` (or a process group)
    # in a one-process-per-GPU job where EVERY rank holds the same chain (same data, same
    # rng seed) and calls `posterior` in lockstep; the n sampled models are then split
    # across the ranks.  Never inferred from the world size: a call on a subset of ranks,
    # or chains that differ per rank (rng=None), would hang or mix different posteriors.
    sharded = False

    def __init__(self, model, prior, n=100, burn=100, rng=None):
        self._model = model.copy()
        self._prior = prior
        self._hypers = np.empty((0, self._model.nhyper))
        self._models = None
        self._batch = None          # (lo, hi, _DeviceBatch of self._hypers[lo:hi]), built on first use
        self._n = n
        self._burn = burn
        self._rng = rstate(rng)
        if self._model.ndata > 0:
            if self._burn > 0:
                sample(self._model, self._prior, self._burn, rng=self._rng)
            self._resample()

    def _resample(self):
        self._hypers = sample(self._model, self._prior, self._n, raw=True, rng=self._rng)
        self._models = None
        self._batch = None

    @property
    def _samples(self):
        """List of model copies, one per sampled hyper vector (built lazily)."""
        if self._models is None:
            self._models = [self._model.copy(h) for h in self._hypers]
        return self._models

    def __iter__(self):
        return iter(self._samples)

    @property
    def ndata(self):
        return self._model.ndata

    @property
    def data(self):
        return self._model.data

    def __deepcopy__(self, memo):
        # the device batch is not cloned: the copy builds its own on first use
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            setattr(new, k, None if k == '_batch' else copy.deepcopy(v, memo))
        return new

    def add_data(self, X, y):
        self._batch = None
        nprev = self._model.ndata
        self._model.add_data(X, y)
        if self._model.ndata > 2*nprev and self._burn > 0:
            sample(self._model, self._prior, self._burn, rng=self._rng)
        self._resample()

    def _device_batch(self, lo, hi):
        """The resident batch of the sampled models lo..hi-1 of an ExactGP chain with data, or None."""
        model = self._model
        if not (isinstance(model, ExactGP) and model.ndata > 0 and len(self._hypers) > 0):
            return None
        if self._batch is None or self._batch[:2] != (lo, hi):
            self._batch = None
            self._batch = (lo, hi, _DeviceBatch(model, self._hypers[lo:hi]))
        return self._batch[2]

    def posterior(self, X, grad=False):
        """Moment-matched mixture over the sampled models (mcmc.py:75-93)."""
        from .. import sharding
        model = self._model
        batched = isinstance(model, ExactGP) and model.ndata > 0 and len(self._hypers) > 0
        if not batched:
            # other models (FITC, DTC) and the prior: one posterior per materialised model
            parts = [m.posterior(X, grad) for m in self._samples]
            return _mixture(*(np.array([p[i] for p in parts]) for i in range(4 if grad else 2)))
        X = model._kernel.transform(X)
        group = None if self.sharded is True else self.sharded
        rank, size = sharding.world(group) if self.sharded else (0, 1)
        if size > 1:
            # one process per GPU, identical chains (same rng) on every rank: the
            # n sampled models are split across the ranks (SURVEY.md 8e), each rank
            # predicting from the resident batch of its slice
            lo, hi = sharding.shard_range(len(self._hypers), rank, size)
            return sharding.sharded_mixture_posterior(
                model, self._hypers, X, group, local_fn=lambda h, x: self._device_batch(lo, hi).predict(x, grad),
                grad=grad)
        return _mixture(*self._device_batch(0, len(self._hypers)).predict(X, grad))
