"""CPU checks of the incremental FITC / DTC update's algebra (tests/fitc_inc_model.py,
the numpy model of pgp_fitc_append_inc): the rank-m Cholesky update with riding
rows, and sequences of appends against the oracle's full FITC / DTC on the same
data."""

import numpy as np
import numpy.testing as nt
import pytest
import scipy.linalg as sla

from oracle.pygp_oracle import make_kernel, OFITC, ODTC
import fitc_inc_model as im

SN, MEAN = 0.1, 0.3


def spd_factor(n, rng):
    B = rng.randn(n, n)
    return np.linalg.cholesky(B.dot(B.T)/n + np.eye(n))


@pytest.mark.parametrize('n', [1, 5, 64, 65, 130])
@pytest.mark.parametrize('m', [1, 3, 7])
def test_chol_update(n, m):
    rng = np.random.RandomState(n*100 + m)
    L = spd_factor(n, rng)
    G = rng.randn(2, n)                      # right-hand sides g_r
    Z = sla.solve_triangular(L, G.T, lower=True).T
    W, C = rng.randn(m, n), rng.randn(m, 2)
    L2, Z2 = im.chol_update(L, Z, W, C)
    ref = np.linalg.cholesky(L.dot(L.T) + W.T.dot(W))
    nt.assert_allclose(L2, ref, rtol=0, atol=1e-12*np.abs(ref).max())
    assert np.all(np.diag(L2) > 0)
    zref = np.linalg.solve(ref, (G + C.T.dot(W)).T).T       # L'^-1 (g + W^T c)
    nt.assert_allclose(Z2, zref, rtol=0, atol=1e-12*np.abs(zref).max())


def wide_range(rng, shape, lo=-165.0):
    """Entries with magnitudes spread from 10^lo to 1 and random signs."""
    return np.sign(rng.randn(*shape))*10.0**rng.uniform(lo, 0.0, size=shape)


def test_chol_update_tiny_pivot():
    """A pivot entry of x far below L_kk (|x|^2 below the smallest double) is
    scaled away before anything of order 1/|x| could form."""
    L = np.eye(3)
    W = np.array([[1e-157, 1.0, 0.5]])
    L2, Z2 = im.chol_update(L, np.zeros((1, 3)), W, np.ones((1, 1)))
    ref = np.linalg.cholesky(np.eye(3) + W.T.dot(W))
    assert np.all(np.isfinite(L2)) and np.all(np.isfinite(Z2))
    nt.assert_allclose(L2, ref, rtol=0, atol=1e-15)
    nt.assert_allclose(Z2[0], np.linalg.solve(ref, W[0]), rtol=0, atol=1e-15)


@pytest.mark.parametrize('n', [5, 65, 130])
@pytest.mark.parametrize('m', [1, 3, 7])
def test_chol_update_wide_range(n, m):
    """Update vectors whose entries span 1e-165 .. 1."""
    rng = np.random.RandomState(7*n + m)
    L = spd_factor(n, rng)
    G = rng.randn(2, n)
    Z = sla.solve_triangular(L, G.T, lower=True).T
    W, C = wide_range(rng, (m, n)), wide_range(rng, (m, 2))
    L2, Z2 = im.chol_update(L, Z, W, C)
    assert np.all(np.isfinite(L2)) and np.all(np.isfinite(Z2))
    ref = np.linalg.cholesky(L.dot(L.T) + W.T.dot(W))
    nt.assert_allclose(L2, ref, rtol=0, atol=1e-12*np.abs(ref).max())
    zref = np.linalg.solve(ref, (G + C.T.dot(W)).T).T
    nt.assert_allclose(Z2, zref, rtol=0, atol=1e-12*np.abs(zref).max())


@pytest.mark.parametrize('ell', [0.02, 0.03])
@pytest.mark.parametrize('dtc', [False, True])
def test_appends_short_length_scale(ell, dtc):
    """SE with 196 pseudo-inputs on a grid and length-scales of a few hundredths:
    the new rows' kernel values reach 1e-160 and below, and one-row appends
    still equal the full update on all the data."""
    k = make_kernel(('se', 1.0, ell, 2))
    g = np.linspace(0, 1, 14)
    U = np.array([(a, b) for a in g for b in g])
    rng = np.random.RandomState(3)
    X = rng.rand(90, 2)
    y = np.sin(3*X.sum(1)) + SN*rng.randn(90)
    st = im.sparse_update(k, SN**2, MEAN, U, X[:40], y[:40], dtc)
    for i in range(40, 90):
        st = im.sparse_append(k, st, U, X[i:i+1], y[i:i+1])
        assert np.all(np.isfinite(st['R'])) and np.all(np.isfinite(st['A']))
    full = im.sparse_update(k, SN**2, MEAN, U, X, y, dtc)
    nt.assert_allclose(im.sparse_lz(st), im.sparse_lz(full), rtol=1e-12)
    Xs = rng.rand(7, 2)
    for a, b in zip(im.sparse_predict(k, st, U, Xs), im.sparse_predict(k, full, U, Xs)):
        nt.assert_allclose(a, b, rtol=0, atol=1e-12*np.abs(b).max())


def problem(d, p, n, seed):
    rng = np.random.RandomState(seed)
    X = rng.rand(n, d)
    y = np.sin(3*X.sum(1)) + SN*rng.randn(n)
    U = rng.rand(p, d)
    Xs = rng.rand(7, d)
    return X, y, U, Xs


CASES = {
    'se_ard3': (('se', 1.0, [0.3, 0.4, 0.5]), 3),
    'matern3_2d': (('matern', 0.8, [0.3, 0.25], 3), 2),
    'se_plus_rq': (('sum', ('se', 1.0, 0.25, 2), ('rq', 0.5, [0.2, 0.3], 0.7)), 2),
}


@pytest.mark.parametrize('name', sorted(CASES))
@pytest.mark.parametrize('dtc', [False, True])
def test_appends_vs_oracle(name, dtc):
    """A model grown by 1-row, 3-row and 8-row appends equals the oracle's full
    FITC / DTC on all the data: lZ, posterior, and the riding rows (beta, b)
    equal direct solves with the updated factors."""
    spec, d = CASES[name]
    k = make_kernel(spec)
    X, y, U, Xs = problem(d, 12, 80, 7)
    n0 = 40
    st = im.sparse_update(k, SN**2, MEAN, U, X[:n0], y[:n0], dtc)
    steps = [1]*5 + [3, 8]
    i = n0
    for m in steps:
        st = im.sparse_append(k, st, U, X[i:i+m], y[i:i+m])
        i += m
    gp = (ODTC if dtc else OFITC)(SN, k, MEAN, U)
    gp.add_data(X[:i], y[:i])
    nt.assert_allclose(im.sparse_lz(st), gp.loglikelihood(), rtol=1e-12)
    mu, s2 = im.sparse_predict(k, st, U, Xs)
    omu, os2 = gp.posterior(Xs)
    nt.assert_allclose(mu, omu, rtol=1e-12, atol=1e-12*np.abs(omu).max())
    nt.assert_allclose(s2, os2, rtol=1e-12, atol=1e-12*np.abs(os2).max())
    # riding rows against direct solves with the updated factors
    beta = sla.solve_triangular(st['A'], st['Vs'].T.dot(st['rs']), lower=True)
    nt.assert_allclose(st['beta'], beta, rtol=0, atol=1e-12*np.abs(beta).max())
    Kxu = k.get(X[:i], U)
    g = Kxu.T.dot(y[:i] - MEAN) if dtc else Kxu.T.dot((y[:i] - MEAN)/st['ell']**2)
    b = sla.solve_triangular(st['R'], g, lower=True)
    nt.assert_allclose(st['b'], b, rtol=0, atol=1e-12*np.abs(b).max())
    # and the factors themselves against a full update on all the data
    full = im.sparse_update(k, SN**2, MEAN, U, X[:i], y[:i], dtc)
    for key in ('A', 'R'):
        nt.assert_allclose(st[key], full[key], rtol=0, atol=1e-12*np.abs(full[key]).max())
