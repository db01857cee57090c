"""Incremental FITC / DTC add_data on the device (pgp_fitc_append_inc) and its
rank-m Cholesky update kernel (pgp_dev_chol_update): a model grown by appends
equals a model built on all the data at once.  Tolerances: 1e-10 relative on
lZ / mu / s2 and 1e-8 on gradients, widened where the numpy model of the same
update (tests/fitc_inc_model.py) shows a larger reordering floor."""

import numpy as np
import numpy.testing as nt
import pytest

from oracle.pygp_oracle import make_kernel
from gpu_util import product_kernel, assert_grad_close
import fitc_inc_model as im

pytestmark = pytest.mark.gpu

SN, MEAN = 0.1, 0.3


def _lib():
    from pygp_b200 import _lib
    return _lib, _lib.context(), _lib.lib()


def kinc():
    return _lib()[2].pgp_fitc_inc_max_rows()


@pytest.mark.parametrize('p', [1, 63, 64, 65, 200, 2048])
@pytest.mark.parametrize('m', [1, 2, 7, 'max'])
@pytest.mark.parametrize('extra', [0, 1])
def test_chol_update_kernel(p, m, extra):
    import torch
    import scipy.linalg as sla
    _, ctx, L = _lib()
    m = kinc() if m == 'max' else m
    rng = np.random.RandomState(p*10 + m + extra)
    B = rng.randn(p, p + 8)
    K = B.dot(B.T)/(p + 8) + 0.5*np.eye(p)
    Lf = np.linalg.cholesky(K)
    G = rng.randn(extra, p)
    ld, ldw = (p + 15)//16*16, (p + extra + 15)//16*16
    F = np.full((p + extra, ld), np.nan)
    F[:p, :p] = Lf + np.triu(np.full((p, p), 7.0), 1)              # the strict upper triangle is left alone
    F[p:, :p] = sla.solve_triangular(Lf, G.T, lower=True).T if extra else 0
    W = np.zeros((m, ldw))
    W[:, :p + extra] = rng.randn(m, p + extra)*0.5
    dF, dW = torch.tensor(F, device='cuda'), torch.tensor(W, device='cuda')
    torch.cuda.synchronize()
    assert L.pgp_dev_chol_update(ctx.handle, dF.data_ptr(), p, ld, extra, dW.data_ptr(), ldw, m) == 0
    out = dF.cpu().numpy()
    ref = np.linalg.cholesky(K + W[:, :p].T.dot(W[:, :p]))
    nt.assert_allclose(np.tril(out[:p, :p]), ref, rtol=0, atol=1e-12*np.abs(ref).max())
    nt.assert_array_equal(np.triu(out[:p, :p], 1), np.triu(F[:p, :p], 1))
    if extra:
        g2 = G + W[:, p:p + extra].T.dot(W[:, :p])
        z = sla.solve_triangular(ref, g2.T, lower=True).T
        nt.assert_allclose(out[p:, :p], z, rtol=0, atol=1e-12*np.abs(z).max())


@pytest.mark.parametrize('p', [1, 65, 200, 2048])
@pytest.mark.parametrize('m', [1, 7, 'max'])
def test_chol_update_kernel_wide_range(p, m):
    """Update vectors and coefficients whose entries span 1e-165 .. 1 (kernel values of
    points many length-scales apart): the reflectors are scaled, nothing overflows."""
    import torch
    import scipy.linalg as sla
    _, ctx, L = _lib()
    m = kinc() if m == 'max' else m
    rng = np.random.RandomState(p + 3*m)
    B = rng.randn(p, p + 8)
    K = B.dot(B.T)/(p + 8) + 0.5*np.eye(p)
    Lf = np.linalg.cholesky(K)
    G = rng.randn(1, p)
    ld, ldw = (p + 15)//16*16, (p + 1 + 15)//16*16
    F = np.zeros((p + 1, ld))
    F[:p, :p] = Lf
    F[p, :p] = sla.solve_triangular(Lf, G[0], lower=True)
    W = np.zeros((m, ldw))
    W[:, :p + 1] = np.sign(rng.randn(m, p + 1))*10.0**rng.uniform(-165, 0, size=(m, p + 1))
    dF, dW = torch.tensor(F, device='cuda'), torch.tensor(W, device='cuda')
    torch.cuda.synchronize()
    assert L.pgp_dev_chol_update(ctx.handle, dF.data_ptr(), p, ld, 1, dW.data_ptr(), ldw, m) == 0
    out = dF.cpu().numpy()
    assert np.all(np.isfinite(out))
    ref = np.linalg.cholesky(K + W[:, :p].T.dot(W[:, :p]))
    nt.assert_allclose(np.tril(out[:p, :p]), ref, rtol=0, atol=1e-12*np.abs(ref).max())
    z = sla.solve_triangular(ref, G[0] + W[:, p].dot(W[:, :p]), lower=True)
    nt.assert_allclose(out[p, :p], z, rtol=0, atol=1e-12*np.abs(z).max())


@pytest.mark.parametrize('dtc', [False, True])
def test_grown_short_length_scale(dtc):
    """SE with 196 pseudo-inputs on a grid and length-scale 0.02: the new rows' kernel
    values reach 1e-160 and below; 50 one-row appends equal a fresh model."""
    import pygp_b200 as pygp
    cls = pygp.inference.DTC if dtc else pygp.inference.FITC
    spec = ('se', 1.0, 0.02, 2)
    g = np.linspace(0, 1, 14)
    U = np.array([(a, b) for a in g for b in g])
    rng = np.random.RandomState(3)
    X = rng.rand(90, 2)
    y = np.sin(3*X.sum(1)) + SN*rng.randn(90)
    Xs = rng.rand(9, 2)
    gp = model(cls, spec, U, X[:40], y[:40])
    h = gp._dev
    for i in range(40, 90):
        gp.add_data(X[i:i + 1], y[i:i + 1])
    assert gp._dev is h
    ref = model(cls, spec, U, X, y)
    lZ, dlZ = gp.loglikelihood(True)
    rlZ, rdlZ = ref.loglikelihood(True)
    assert np.isfinite(lZ) and np.all(np.isfinite(dlZ))
    nt.assert_allclose(lZ, rlZ, rtol=1e-10)
    assert_grad_close(dlZ, rdlZ)
    mu, s2 = gp.posterior(Xs)
    rmu, rs2 = ref.posterior(Xs)
    nt.assert_allclose(mu, rmu, rtol=1e-10, atol=1e-10*np.abs(rmu).max())
    nt.assert_allclose(s2, rs2, rtol=1e-10, atol=1e-10*np.abs(rs2).max())


def test_chol_update_rejects_too_many_rows():
    import torch
    _, ctx, L = _lib()
    m = kinc() + 1
    F = np.eye(4, 16)
    dF, dW = torch.tensor(F, device='cuda'), torch.zeros((m, 16), dtype=torch.float64, device='cuda')
    torch.cuda.synchronize()
    assert L.pgp_dev_chol_update(ctx.handle, dF.data_ptr(), 4, 16, 0, dW.data_ptr(), 16, m) == -1
    nt.assert_array_equal(dF.cpu().numpy(), F)


CASES = {
    'se_ard8_p128': (('se', 1.0, [0.7]*8), 8, 128),
    'matern5_p65': (('matern', 0.8, [0.35, 0.3, 0.4], 5), 3, 65),
    'se_plus_rq': (('sum', ('se', 1.0, 0.25, 2), ('rq', 0.5, [0.2, 0.3], 0.7)), 2, 40),
}


def problem(d, p, n, seed=3):
    rng = np.random.RandomState(seed)
    X = rng.rand(n, d)
    y = np.sin(3*X.sum(1)) + SN*rng.randn(n)
    U = rng.rand(p, d)
    Xs = rng.rand(9, d)
    return X, y, U, Xs


def model(cls, spec, U, X, y):
    import pygp_b200 as pygp
    gp = cls(pygp.likelihoods.Gaussian(SN), product_kernel(spec), MEAN, U)
    gp.add_data(X, y)
    return gp


def steps():
    return [1]*50 + [7, kinc()]


def grow(cls, spec, U, X, y, n0):
    """Build on the first n0 rows, then append the rest by the steps; every append
    must keep the device handle (the incremental path)."""
    gp = model(cls, spec, U, X[:n0], y[:n0])
    gp.loglikelihood(True)                  # gradient buffers allocated at the first capacity
    h = gp._dev
    i = n0
    for m in steps():
        gp.add_data(X[i:i + m], y[i:i + m])
        assert gp._dev is h
        i += m
    return gp


def model_floor(spec, U, X, y, Xs, n0, dtc):
    """|incremental - full| of the numpy model for mu and s2 (the reordering floor)."""
    k = make_kernel(spec)
    st = im.sparse_update(k, SN**2, MEAN, U, X[:n0], y[:n0], dtc)
    i = n0
    for m in steps():
        st = im.sparse_append(k, st, U, X[i:i + m], y[i:i + m])
        i += m
    full = im.sparse_update(k, SN**2, MEAN, U, X, y, dtc)
    a, b = im.sparse_predict(k, st, U, Xs), im.sparse_predict(k, full, U, Xs)
    return np.abs(a[0] - b[0]).max(), np.abs(a[1] - b[1]).max()


@pytest.mark.parametrize('name', sorted(CASES))
@pytest.mark.parametrize('dtc', [False, True])
@pytest.mark.parametrize('n0', [70, 300])
def test_grown_equals_fresh(name, dtc, n0):
    import pygp_b200 as pygp
    cls = pygp.inference.DTC if dtc else pygp.inference.FITC
    spec, d, p = CASES[name]
    n = n0 + sum(steps())
    X, y, U, Xs = problem(d, p, n)
    gp = grow(cls, spec, U, X, y, n0)
    ref = model(cls, spec, U, X, y)
    assert gp.ndata == ref.ndata == n
    fmu, fs2 = model_floor(spec, U, X, y, Xs, n0, dtc)

    lZ, dlZ, dU = gp.loglikelihood(True, pseudoinputs=True)
    rlZ, rdlZ, rdU = ref.loglikelihood(True, pseudoinputs=True)
    assert gp.loglikelihood() == lZ
    nt.assert_allclose(lZ, rlZ, rtol=1e-10)
    assert_grad_close(dlZ, rdlZ)
    assert_grad_close(dU, rdU)

    mu, s2, dmu, ds2 = gp.posterior(Xs, grad=True)
    rmu, rs2, rdmu, rds2 = ref.posterior(Xs, grad=True)
    nt.assert_allclose(mu, rmu, rtol=1e-10, atol=max(1e-10*np.abs(rmu).max(), 10*fmu))
    nt.assert_allclose(s2, rs2, rtol=1e-10, atol=max(1e-10*np.abs(rs2).max(), 10*fs2))
    assert_grad_close(dmu, rdmu)
    assert_grad_close(ds2, rds2)

    m, S = gp._full_posterior(Xs)
    rm, rS = ref._full_posterior(Xs)
    nt.assert_allclose(m, rm, rtol=1e-10, atol=max(1e-10*np.abs(rm).max(), 10*fmu))
    nt.assert_allclose(S, rS, rtol=1e-10, atol=max(1e-10*np.abs(rS).max(), 10*fs2))


@pytest.mark.parametrize('dtc', [False, True])
def test_set_hyper_copy_and_pseudoinputs_after_appends(dtc):
    import pygp_b200 as pygp
    cls = pygp.inference.DTC if dtc else pygp.inference.FITC
    spec, d, p = CASES['matern5_p65']
    n0 = 90
    n = n0 + sum(steps())
    X, y, U, Xs = problem(d, p, n, seed=5)
    gp = grow(cls, spec, U, X, y, n0)

    # copy() of an appended model rebuilds its device state and is usable
    c = gp.copy()
    nt.assert_allclose(c.loglikelihood(), gp.loglikelihood(), rtol=1e-10)
    nt.assert_allclose(c.posterior(Xs)[0], gp.posterior(Xs)[0], rtol=1e-10, atol=1e-10)

    # set_hyper refactors the grown handle and equals a fresh model at those hypers
    h = gp.get_hyper() + 0.1
    gp.set_hyper(h)
    ref = model(cls, spec, U, X, y)
    ref.set_hyper(h)
    lZ, dlZ = gp.loglikelihood(True)
    rlZ, rdlZ = ref.loglikelihood(True)
    nt.assert_allclose(lZ, rlZ, rtol=1e-12)
    assert_grad_close(dlZ, rdlZ, rtol=1e-10)
    nt.assert_allclose(gp.posterior(Xs), ref.posterior(Xs), rtol=1e-12, atol=1e-12)

    # after set_pseudoinputs the next add_data takes the full path and equals a fresh model
    U2 = U + 0.01
    gp._set_pseudoinputs(U2)
    Xa, ya = np.random.RandomState(9).rand(3, d), np.array([0.1, -0.2, 0.3])
    h_dev = gp._dev
    gp.add_data(Xa, ya)
    assert gp._dev is not h_dev
    ref2 = model(cls, spec, U2, np.r_[X, Xa], np.r_[y, ya])
    ref2.set_hyper(h)
    nt.assert_allclose(gp.loglikelihood(), ref2.loglikelihood(), rtol=1e-12)
    nt.assert_allclose(gp.posterior(Xs), ref2.posterior(Xs), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize('dtc', [False, True])
def test_path_selection(dtc):
    """Up to min(ndata, kIncRows) rows go incremental (same handle); more replace it."""
    import pygp_b200 as pygp
    cls = pygp.inference.DTC if dtc else pygp.inference.FITC
    spec, d, p = CASES['se_plus_rq']
    X, y, U, Xs = problem(d, p, 400, seed=11)
    gp = model(cls, spec, U, X[:30], y[:30])
    h = gp._dev
    gp.add_data(X[30:60], y[30:60])             # 30 onto 30: incremental
    assert gp._dev is h and gp._ndev == 60
    gp.add_data(X[60:121], y[60:121])           # 61 onto 60: more than ndata -> full update
    assert gp._dev is not h and gp._ndev == 121
    h = gp._dev
    k = kinc()
    gp.add_data(X[121:121 + k], y[121:121 + k])     # kIncRows onto 121: incremental
    assert gp._dev is h
    i = 121 + k
    gp.add_data(X[i:i + k + 1], y[i:i + k + 1])     # kIncRows + 1: full update
    assert gp._dev is not h
    i += k + 1
    ref = model(cls, spec, U, X[:i], y[:i])
    nt.assert_allclose(gp.loglikelihood(), ref.loglikelihood(), rtol=1e-10)
