"""Pseudo-input gradient of the FITC / DTC log marginal likelihood
(pgp_fitc_loglike_pseudo, gram.cu pseudo_gram_kernel), moving the pseudo-inputs
(FITC.set_pseudoinputs) and fitting them (learning.optimize(pseudoinputs=True)).

The numpy model (oracle/fitc_pseudo.py) is checked against central differences
of the oracle's lZ on the CPU; the device against the model and against central
differences of its own lZ on the GPU."""

import os
import re

import numpy as np
import numpy.testing as nt
import pytest

from oracle import fitc_model as fm
from oracle import fitc_pseudo as fp
from oracle.pygp_oracle import make_kernel, synthetic_problem
from gpu_util import product_kernel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KERNELS = [
    (('se', 1.0, 0.4, 2), 2),
    (('se', 1.0, [0.5, 0.7]), 2),
    (('matern', 1.0, 0.5, 1, 1), 1),
    (('matern', 1.0, [0.6, 0.4], 3), 2),
    (('matern', 0.9, [0.5, 0.6], 5), 2),
    (('rq', 0.8, [0.5, 0.6], 0.7), 2),
    (('periodic', 1.0, 0.5, 0.7), 1),
    (('sum', ('se', 1.0, [0.3, 0.4]), ('rq', 0.5, [0.6, 0.5], 0.8)), 2),
    (('prod', ('se', 1.0, [0.5, 0.6]), ('matern', 1.0, [0.7, 0.8], 5)), 2),
]
KID = [s[0] + ('-iso' if not isinstance(s[2], list) and s[0] in ('se', 'matern') else '') for s, _ in KERNELS]


def model_lz_grad(k, U, X, y, dtc, sn2=0.09, mean=0.1):
    if dtc:
        st = fm.dtc_update(k, sn2, mean, U, X, y)
        return fm.dtc_loglike(k, st, U, X), fp.dtc_pseudo_grad(k, st, U, X)
    st = fm.fitc_update(k, sn2, mean, U, X, y)
    return fm.fitc_loglike(k, st, U, X), fp.fitc_pseudo_grad(k, st, U, X)


def central_differences(lz, U, h):
    fd = np.zeros_like(U)
    for j in range(U.shape[0]):
        for k in range(U.shape[1]):
            Up, Um = U.copy(), U.copy()
            Up[j, k] += h
            Um[j, k] -= h
            fd[j, k] = (lz(Up) - lz(Um)) / (2*h)
    return fd


# ---- CPU: the model against central differences of the oracle's lZ ------------------------------------
@pytest.mark.parametrize('dtc', [False, True], ids=['fitc', 'dtc'])
@pytest.mark.parametrize('spec,d', KERNELS, ids=KID)
def test_model_vs_central_differences(spec, d, dtc):
    """h = 1e-6 for every kernel: Periodic's truncation error at h = 1e-4 is 5e-6 of max|dU|."""
    k = make_kernel(spec)
    rng = np.random.RandomState(0)
    X = rng.rand(60, d)
    y = np.sin(4*X.sum(1)) + 0.1*rng.randn(60)
    U = rng.rand(7, d)
    _, g = model_lz_grad(k, U, X, y, dtc)
    fd = central_differences(lambda V: model_lz_grad(k, V, X, y, dtc)[0], U, 1e-6)
    assert g.shape == U.shape
    nt.assert_allclose(g, fd, rtol=0, atol=1e-6*np.abs(fd).max())


def test_set_pseudoinputs_checks_columns():
    import pygp_b200 as pygp
    gp = pygp.inference.FITC(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [0.5, 0.6]), 0.0, np.zeros((4, 2)))
    with pytest.raises(ValueError):
        gp.set_pseudoinputs(np.zeros((4, 3)))
    with pytest.raises(ValueError):
        pygp.inference.DTC.from_gp(gp).set_pseudoinputs(np.zeros(4))
    U = np.ones((5, 2))
    gp.set_pseudoinputs(U)                     # no data: nothing on the device
    U[0, 0] = 7.0
    assert gp.pseudoinputs.shape == (5, 2) and gp.pseudoinputs[0, 0] == 1.0


def test_optimize_pseudoinputs_needs_pseudoinputs():
    import pygp_b200 as pygp
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, 0.5), 0.0)
    with pytest.raises(ValueError):
        pygp.optimize(gp, pseudoinputs=True)


def test_pseudo_kernel_does_not_spill():
    """-Xptxas -v of gram.cu: no instantiation of the contraction kernel spills to local memory."""
    import __graft_entry__ as g
    g.build()
    log = open(os.path.join(ROOT, 'pygp_b200', 'csrc', 'build', 'gram.ptxas.log')).read()
    blocks = re.findall(r"Compiling entry function '(\w*pseudo_gram_kernel\w*)'[^\n]*\n[^\n]*Function properties[^\n]*\n"
                        r"([^\n]*)\n([^\n]*)\n", log)
    assert len(blocks) >= 7, 'one instantiation per leaf type and the composite expected'
    for name, props, regs in blocks:
        assert '0 bytes spill stores, 0 bytes spill loads' in props, (name, props)
        assert int(re.search(r'Used (\d+) registers', regs).group(1)) <= 128, (name, regs)


# ---- GPU ----------------------------------------------------------------------------------------------
def device_model(spec, U, X, y, dtc, sn=0.1, mean=0.1):
    import pygp_b200 as pygp
    cls = pygp.inference.DTC if dtc else pygp.inference.FITC
    gp = cls(pygp.likelihoods.Gaussian(sn), product_kernel(spec), mean, U)
    gp.add_data(X, y)
    return gp


MEDIUM = [
    (('se', 1.0, [0.5*np.sqrt(8)]*8), 3000, 8, 128),
    (('matern', 1.0, [0.8, 0.9, 0.7], 5), 5001, 3, 65),
    (('sum', ('se', 1.0, [0.15, 0.2]), ('rq', 0.5, [0.2, 0.25], 0.8)), 1200, 2, 96),
    (('se', 1.0, 0.05, 1), 70000, 1, 33),
    (('matern', 1.0, [0.9, 1.1, 0.8, 1.0, 1.2], 3), 2000, 5, 40),
    (('se', 1.0, [1.2]*12), 1500, 12, 70),
]


@pytest.mark.gpu
@pytest.mark.parametrize('dtc', [False, True], ids=['fitc', 'dtc'])
@pytest.mark.parametrize('spec,N,d,p', MEDIUM, ids=['se-ard8', 'm5-ragged', 'se+rq', '1d-70000', 'm3-d5-p40', 'se-d12'])
def test_vs_model(spec, N, d, p, dtc):
    """Device dU against the numpy model at the shapes of test_fitc_gpu.py::test_vs_oracle_medium, plus
    p < 64 with d = 5 and d = 12 (two groups of eight input dimensions).  The floor of the tolerance is
    the model's own sensitivity to the order of its float64 arithmetic, measured as in that test: the
    model evaluated again with the data and the pseudo-inputs permuted (chol(Kuu + su2 I) has condition
    numbers up to 1e9 here)."""
    X, y, _ = synthetic_problem(N, d, 0)
    U = np.random.RandomState(3).rand(p, d) if d > 1 else np.linspace(0, 1, p)[:, None]
    gp = device_model(spec, U, X, y, dtc)
    lZ0, dlZ0 = gp.loglikelihood(True)
    lZ, dlZ, dU = gp.loglikelihood(True, pseudoinputs=True)
    assert lZ == lZ0 and np.array_equal(dlZ, dlZ0)           # bitwise those of loglikelihood(True)
    assert np.array_equal(gp.loglikelihood(True, pseudoinputs=True)[2], dU)
    assert dU.shape == U.shape
    ok = make_kernel(spec)
    _, m = model_lz_grad(ok, U, X, y, dtc, sn2=0.01)
    pu, px = np.random.RandomState(5).permutation(p), np.random.RandomState(6).permutation(N)
    _, mp = model_lz_grad(ok, U[pu], X[px], y[px], dtc, sn2=0.01)
    mp = mp[np.argsort(pu)]
    sens = 20*float(np.abs(m - mp).max())
    nt.assert_allclose(dU, m, rtol=0, atol=max(1e-8*np.abs(m).max(), sens))


SMALL = [
    (('se', 1.0, [0.5, 0.6]), 2),
    (('matern', 1.0, 0.5, 1, 1), 1),
    (('matern', 1.0, [0.6, 0.5], 3), 2),
    (('matern', 1.0, [0.6, 0.7], 5), 2),
    (('rq', 0.8, [0.5, 0.6], 0.7), 2),
    (('periodic', 1.0, 0.5, 0.7), 1),
    (('prod', ('se', 1.0, 0.5, 1), ('periodic', 1.0, 0.8, 0.9)), 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize('dtc', [False, True], ids=['fitc', 'dtc'])
@pytest.mark.parametrize('spec,d', SMALL, ids=['se', 'm1', 'm3', 'm5', 'rq', 'periodic', 'se*per'])
def test_vs_device_differences(spec, d, dtc):
    """Central differences (h = 1e-5) of the device's own lZ, U moved through set_pseudoinputs."""
    rng = np.random.RandomState(1)
    X = rng.rand(300, d)
    y = np.sin(4*X.sum(1)) + 0.1*rng.randn(300)
    U = rng.rand(9, d)
    gp = device_model(spec, U, X, y, dtc, sn=0.3)
    _, _, dU = gp.loglikelihood(True, pseudoinputs=True)

    def lz(V):
        gp.set_pseudoinputs(V)
        return gp.loglikelihood()
    fd = central_differences(lz, U, 1e-5)
    nt.assert_allclose(dU, fd, rtol=0, atol=1e-5*np.abs(fd).max())


@pytest.mark.gpu
@pytest.mark.parametrize('dtc', [False, True], ids=['fitc', 'dtc'])
def test_set_pseudoinputs(dtc):
    import pygp_b200 as pygp
    X, y, Xs = synthetic_problem(800, 2, 50)
    spec = ('se', 1.0, [0.4, 0.5])
    U = np.random.RandomState(3).rand(24, 2)
    U2 = np.random.RandomState(4).rand(24, 2)
    gp = device_model(spec, U, X, y, dtc)
    c = gp.copy()
    gp.set_pseudoinputs(U2)
    c.set_pseudoinputs(U2)
    fresh = device_model(spec, U2, X, y, dtc)
    lZ, dlZ = fresh.loglikelihood(True)
    mu, s2 = fresh.posterior(Xs)
    for g in (gp, c):
        nt.assert_allclose(g.pseudoinputs, U2, rtol=0)
        l, dl = g.loglikelihood(True)
        nt.assert_allclose(l, lZ, rtol=1e-12)
        nt.assert_allclose(dl, dlZ, rtol=1e-12, atol=1e-12*np.abs(dlZ).max())
        m, s = g.posterior(Xs)
        nt.assert_allclose(m, mu, rtol=1e-12, atol=1e-12*np.abs(mu).max())
        nt.assert_allclose(s, s2, rtol=1e-12, atol=1e-12*np.abs(s2).max())
    # a different number of pseudo-inputs rebuilds the device state
    U3 = np.random.RandomState(5).rand(31, 2)
    gp.set_pseudoinputs(U3)
    f3 = device_model(spec, U3, X, y, dtc)
    nt.assert_allclose(gp.loglikelihood(), f3.loglikelihood(), rtol=1e-12)
    assert gp.loglikelihood(True, pseudoinputs=True)[2].shape == (31, 2)
    with pytest.raises(ValueError):
        gp.set_pseudoinputs(np.zeros((31, 3)))
    # moved without a factorisation: the state refuses a gradient until the next update
    gp._set_pseudoinputs(U3 + 0.01)
    with pytest.raises(RuntimeError):
        gp.loglikelihood(True, pseudoinputs=True)


@pytest.mark.gpu
def test_loglike_pseudo_before_update_raises():
    import ctypes as C
    from pygp_b200 import _lib
    from pygp_b200.inference.fitc import _DeviceFITC
    import pygp_b200 as pygp
    X, y, _ = synthetic_problem(100, 2, 0)
    dev = _DeviceFITC.create(pygp.kernels.SE(1.0, [0.5, 0.5]), X[:8], X, y)
    lZ, dlZ, dU = C.c_double(), np.empty(5), np.empty((8, 2))
    with pytest.raises(RuntimeError):
        _lib.check(dev.ctx, _lib.lib().pgp_fitc_loglike_pseudo(dev.handle, C.byref(lZ), _lib.ptr(dlZ), _lib.ptr(dU)))


def learning_problem():
    rng = np.random.RandomState(0)
    X = rng.rand(200, 1)
    y = np.sin(6*X[:, 0]) + 0.1*rng.randn(200)
    U = np.linspace(0.0, 0.1, 8)[:, None]          # clustered at one end of the data
    return X, y, U


@pytest.mark.gpu
def test_optimize_pseudoinputs(monkeypatch):
    import pygp_b200 as pygp
    from pygp_b200 import _lib
    X, y, U = learning_problem()
    mk = lambda: device_model(('se', 1.0, 0.3, 1), U, X, y, False, sn=0.3, mean=0.0)
    ref = mk()
    pygp.optimize(ref)
    lib = _lib.lib()
    calls = {'pgp_fitc_update': 0, 'pgp_fitc_loglike_pseudo': 0}
    for name in calls:
        fn = getattr(lib, name)

        def counted(*args, _fn=fn, _name=name):
            calls[_name] += 1
            return _fn(*args)
        monkeypatch.setattr(lib, name, counted)
    gp = mk()
    calls['pgp_fitc_update'] = 0
    pygp.optimize(gp, pseudoinputs=True)
    # one factorisation per objective evaluation, one more for the final state
    assert calls['pgp_fitc_loglike_pseudo'] > 1
    assert calls['pgp_fitc_update'] == calls['pgp_fitc_loglike_pseudo'] + 1
    monkeypatch.undo()
    assert gp.loglikelihood() > ref.loglikelihood() + 1.0
    Uf = gp.pseudoinputs[:, 0]
    assert Uf.min() < 0.3 and Uf.max() > 0.7                 # spread over the data in [0, 1]
    _, dlZ, dU = gp.loglikelihood(True, pseudoinputs=True)
    _, dlZ0, dU0 = mk().loglikelihood(True, pseudoinputs=True)
    g, g0 = np.r_[dlZ, dU.ravel()], np.r_[dlZ0, dU0.ravel()]
    assert np.abs(g).max() < 1e-2*np.abs(g0).max(), (np.abs(g).max(), np.abs(g0).max())
