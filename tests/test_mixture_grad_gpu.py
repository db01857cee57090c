"""Resident batches of exact GPs (pgp_batch) and the mixture posterior with
input-gradients on top of them (meta.MCMC.posterior(X, grad=True)):
per-component gradients against single models and the oracle, bitwise
agreement with pgp_batched_predict and between resident and refactored
problems, the MCMC mixture against the loop over its models and finite
differences, and the sharded reduction on one rank."""

import copy

import numpy as np
import numpy.testing as nt
import pytest

from oracle.pygp_oracle import make_kernel, OExactGP, synthetic_problem
from gpu_util import product_kernel, assert_grad_close, assert_pred_close

pytestmark = pytest.mark.gpu

SN = 0.1


def _problem(spec, n, d, ms, B, seed=0):
    import pygp_b200 as pygp
    X, y, Xs = synthetic_problem(n, d, ms, seed=seed)
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(SN), product_kernel(spec), 0.1)
    gp.add_data(X, y)
    H = gp.get_hyper() + np.random.RandomState(seed + 5).uniform(-0.2, 0.2, size=(B, gp.nhyper))
    return gp, H, X, y, Xs


def _batch(gp, H, budget=0):
    from pygp_b200.meta.mcmc import _DeviceBatch
    return _DeviceBatch(gp, H, budget)


CASES = [
    # spec, n, d, ms
    (('se', 1.0, [0.5]), 130, 1, 1),
    (('se', 1.0, [0.3 + 0.05*k for k in range(8)]), 300, 8, 77),
    (('se', 1.0, [0.8 + 0.05*k for k in range(20)]), 201, 20, 65),
    (('matern', 1.0, [0.5, 0.6, 0.7], 1), 157, 3, 70),
    (('matern', 1.0, [0.5, 0.6, 0.7], 3), 157, 3, 1),
    (('matern', 1.0, [0.5, 0.6, 0.7], 5), 157, 3, 129),
    (('matern', 1.0, [0.5, 0.6, 0.7], 5), 157, 3, 12),           # 16 threads per test point
    (('se', 1.0, [0.3 + 0.05*k for k in range(8)]), 300, 8, 20),  # 8 threads per test point
    (('periodic', 0.5, 0.4, 0.3), 150, 1, 33),
    (('rq', 0.5, [0.4, 0.5], 0.3), 140, 2, 66),
    (('rq', 0.5, 0.4, 0.3, 2), 140, 2, 5),
    (('sum', ('se', 1.0, 0.5), ('periodic', 0.5, 1.0, 0.25)), 190, 1, 63),
    (('prod', ('se', 0.8, 0.3, 2), ('matern', 1.0, [0.5, 0.6], 5)), 170, 2, 65),
]


@pytest.mark.parametrize('spec,n,d,ms', CASES, ids=lambda v: None if not isinstance(v, tuple) else v[0])
def test_components_match_single_models(spec, n, d, ms):
    B = 4
    gp, H, X, y, Xs = _problem(spec, n, d, ms, B)
    mu, s2, dmu, ds2 = _batch(gp, H).predict(Xs, grad=True)
    assert dmu.shape == (B, ms, d) and ds2.shape == (B, ms, d)
    for b in range(B):
        m0, v0, dm0, dv0 = gp.copy(H[b]).posterior(Xs, grad=True)
        assert_pred_close(mu[b], s2[b], m0, v0)
        assert_grad_close(dmu[b], dm0)
        assert_grad_close(ds2[b], dv0)
    for b in (0, B - 1):                  # two components against the oracle
        og = OExactGP(SN, make_kernel(spec), 0.1)
        og.add_data(X, y)
        og.set_hyper(H[b])
        m0, v0, dm0, dv0 = og.posterior(Xs, grad=True)
        assert_pred_close(mu[b], s2[b], m0, v0)
        assert_grad_close(dmu[b], dm0)
        assert_grad_close(ds2[b], dv0)


def test_bits():
    from pygp_b200 import sharding
    spec = ('matern', 1.0, [0.5, 0.6, 0.7], 5)
    B = 6
    gp, H, X, y, Xs = _problem(spec, 301, 3, 70, B, seed=2)
    full = _batch(gp, H)
    assert full.resident == B
    ref_mu, ref_s2 = sharding._batched('predict', gp, H, Xs)          # pgp_batched_predict
    mu, s2 = full.predict(Xs)
    nt.assert_array_equal(mu, ref_mu)
    nt.assert_array_equal(s2, ref_s2)
    out = full.predict(Xs, grad=True)
    nt.assert_array_equal(out[0], ref_mu)
    nt.assert_array_equal(out[1], ref_s2)
    again = full.predict(Xs, grad=True)
    for a, b in zip(out, again):
        nt.assert_array_equal(a, b)
    # a budget for 4 of the 6 factors: 3 stay resident, the others are refactored in the remaining slot
    n, ld = 301, 304
    per = 8*((n + 1)*ld + (n//64*64 + 128)*3 + 1) + 8192
    part = _batch(gp, H, budget=int(4.5*per))
    assert 0 < part.resident < B
    got = part.predict(Xs, grad=True)
    for a, b in zip(got, out):
        nt.assert_array_equal(a, b)
    got = part.predict(Xs)
    nt.assert_array_equal(got[0], ref_mu)
    nt.assert_array_equal(got[1], ref_s2)


def test_more_problems_than_one_chunk():
    """B above the 32768 problems of one chunk, all resident: every problem keeps its own factor."""
    from pygp_b200 import sharding
    B = 32769
    gp, H, X, y, Xs = _problem(('se', 1.0, [0.5, 0.6]), 20, 2, 3, B, seed=4)
    bt = _batch(gp, H)
    assert bt.resident == B
    mu, s2, dmu, ds2 = bt.predict(Xs, grad=True)
    ref_mu, ref_s2 = sharding._batched('predict', gp, H, Xs)          # pgp_batched_predict, same chunks
    nt.assert_array_equal(mu, ref_mu)
    nt.assert_array_equal(s2, ref_s2)
    for b in (0, 7, 32767, 32768):
        m0, v0, dm0, dv0 = gp.copy(H[b]).posterior(Xs, grad=True)
        assert_pred_close(mu[b], s2[b], m0, v0)
        assert_grad_close(dmu[b], dm0)
        assert_grad_close(ds2[b], dv0)


def _chain(n=8, seed=0):
    import pygp_b200 as pygp
    ndim = 2
    prior = {'sn': pygp.priors.Uniform(0.01, 1.0), 'sf': pygp.priors.Uniform(0.01, 5.0),
             'ell': pygp.priors.Uniform([0.01]*ndim, [1.0]*ndim),
             'mu': pygp.priors.Uniform([-2.0], [2.0])}
    model = pygp.meta.MCMC(pygp.BasicGP(0.5, 1, [1]*ndim), prior, n=n, burn=0, rng=seed)
    rng = np.random.RandomState(seed)
    model.add_data(rng.rand(40, ndim), rng.rand(40))
    return model, rng


def _loop_mixture(model, X):
    parts = [m.posterior(X, True) for m in model]
    mu_, s2_, dmu_, ds2_ = (np.array([p[i] for p in parts]) for i in range(4))
    mu = np.mean(mu_, axis=0)
    s2 = np.mean(s2_ + (mu_ - mu)**2, axis=0)
    dmu = np.mean(dmu_, axis=0)
    Dmu = dmu_ - dmu
    ds2 = np.mean(ds2_ + 2*mu_[:, :, None]*Dmu - 2*mu[None, :, None]*Dmu, axis=0)
    return mu, s2, dmu, ds2


def test_mcmc_posterior_grad():
    import scipy.optimize as spop
    model, rng = _chain()
    Xq = rng.rand(5, 2)
    out = model.posterior(Xq, grad=True)
    ref = _loop_mixture(model, Xq)
    for a, b in zip(out, ref):
        nt.assert_allclose(a, b, rtol=1e-10, atol=1e-10*max(1.0, np.abs(b).max()))
    again = model.posterior(Xq, grad=True)
    for a, b in zip(out, again):
        nt.assert_array_equal(a, b)
    mu, s2 = model.posterior(Xq)
    nt.assert_array_equal(mu, out[0])
    nt.assert_array_equal(s2, out[1])
    f_mu = lambda x: model.posterior(x[None])[0][0]        # noqa: E731
    f_s2 = lambda x: model.posterior(x[None])[1][0]        # noqa: E731
    nt.assert_allclose(out[2], [spop.approx_fprime(x, f_mu, 1e-7) for x in Xq], rtol=1e-5, atol=1e-5)
    nt.assert_allclose(out[3], [spop.approx_fprime(x, f_s2, 1e-7) for x in Xq], rtol=1e-4, atol=1e-5)
    # a deep copy builds its own batch and gives the same bits
    cp = copy.deepcopy(model)
    assert cp._batch is None
    for a, b in zip(cp.posterior(Xq, grad=True), out):
        nt.assert_array_equal(a, b)


def test_mcmc_add_data_refreshes_the_batch():
    from pygp_b200.meta.mcmc import _DeviceBatch, _mixture
    model, rng = _chain(seed=3)
    Xq = rng.rand(4, 2)
    model.posterior(Xq, grad=True)
    assert model._batch is not None
    model.add_data(rng.rand(7, 2), rng.rand(7))
    assert model._batch is None and model.ndata == 47
    out = model.posterior(Xq, grad=True)
    fresh = _mixture(*_DeviceBatch(model._model, model._hypers).predict(Xq, True))
    for a, b in zip(out, fresh):
        nt.assert_array_equal(a, b)
    ref = _loop_mixture(model, Xq)
    for a, b in zip(out, ref):
        nt.assert_allclose(a, b, rtol=1e-10, atol=1e-10*max(1.0, np.abs(b).max()))


def test_mcmc_not_positive_definite_raises():
    import pygp_b200 as pygp
    X = np.r_[np.linspace(0, 1, 40), np.linspace(0, 1, 40)][:, None]     # duplicated rows
    prior = {'sn': pygp.priors.Uniform(0.01, 1.0), 'sf': pygp.priors.Uniform(0.01, 5.0),
             'ell': pygp.priors.Uniform([0.01], [1.0]), 'mu': pygp.priors.Uniform([-2.0], [2.0])}
    model = pygp.meta.MCMC(pygp.BasicGP(0.5, 1, [0.5]), prior, n=4, burn=0, rng=0)
    model.add_data(X, np.sin(X[:, 0]))
    bad = model._hypers.copy()
    bad[1] = [np.log(1e-12), 0.0, np.log(5.0), 0.0]
    model._hypers, model._batch, model._models = bad, None, None
    with pytest.raises(np.linalg.LinAlgError):
        model.posterior(X[:3], grad=True)
    with pytest.raises(np.linalg.LinAlgError):
        model.posterior(X[:3])


def test_sharded_single_rank_equals_mcmc():
    from pygp_b200 import sharding
    model, rng = _chain(seed=5)
    Xq = rng.rand(6, 2)
    out = model.posterior(Xq, grad=True)
    got = sharding.sharded_mixture_posterior(model._model, model._hypers, Xq, grad=True)
    for a, b in zip(got, out):
        nt.assert_allclose(a, b, rtol=1e-12, atol=1e-14*max(1.0, np.abs(b).max()))
    nt.assert_array_equal(got[0], out[0])
