"""The oracle (oracle/pygp_oracle.py) against the committed reference outputs
(tests/golden, written by oracle/make_golden.py from the unmodified reference),
the known answers of SURVEY.md 8c, and the reference's own self-consistency
checks (tests/test_kernels.py:53-85, tests/test_inference.py:105-112)."""

import numpy as np
import numpy.testing as nt
import pytest
import scipy.optimize as spop

from oracle.cases import (KERNEL_CASES, GP_CASES, DTC_CASES, SURVEY_KAT, GP_SN, GP_MEAN,
                          kernel_inputs, gp_inputs)
from oracle.pygp_oracle import make_kernel, OExactGP, OFITC


@pytest.mark.parametrize('name', sorted(KERNEL_CASES))
def test_kernel_vs_golden(name, golden):
    g = golden['kernels']
    k = make_kernel(KERNEL_CASES[name])
    x1, x2 = kernel_inputs(k.ndim)
    nt.assert_array_equal(k.get_hyper(), g[name + '/hyper'])
    nt.assert_allclose(k.get(x1, x2), g[name + '/get12'], rtol=1e-13, atol=1e-15)
    nt.assert_allclose(k.get(x1), g[name + '/get11'], rtol=1e-13, atol=1e-15)
    nt.assert_allclose(np.array(k.grad(x1, x2)), g[name + '/grad12'], rtol=1e-12, atol=1e-14)
    nt.assert_allclose(np.array(k.grad(x1)), g[name + '/grad11'], rtol=1e-12, atol=1e-14)
    nt.assert_allclose(k.gradx(x1, x2), g[name + '/gradx12'], rtol=1e-12, atol=1e-14)
    nt.assert_allclose(k.grady(x1, x2), g[name + '/grady12'], rtol=1e-12, atol=1e-14)
    nt.assert_allclose(k.gradx(x1), g[name + '/gradx11'], rtol=1e-12, atol=1e-14)
    if name + '/gradxy12' in g.files:
        nt.assert_allclose(k.gradxy(x1, x2), g[name + '/gradxy12'], rtol=1e-11, atol=1e-13)
    else:
        with pytest.raises(NotImplementedError):
            k.gradxy(x1, x2)
    nt.assert_allclose(k.dget(x1), g[name + '/dget'], rtol=1e-15)
    nt.assert_allclose(np.array(k.dgrad(x1)), g[name + '/dgrad'], rtol=1e-15)
    k2 = k.copy_with(g[name + '/hyper2'])
    nt.assert_allclose(k2.get(x1, x2), g[name + '/get12_h2'], rtol=1e-13, atol=1e-15)
    nt.assert_allclose(np.array(k2.grad(x1, x2)), g[name + '/grad12_h2'], rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize('name', sorted(KERNEL_CASES))
def test_kernel_self_consistency(name):
    # tests/test_kernels.py:53-85
    k = make_kernel(KERNEL_CASES[name])
    x1, x2 = kernel_inputs(k.ndim)
    nt.assert_allclose(k.get(x1, x2), k.get(x2, x1).T)
    nt.assert_allclose(np.array(k.grad(x1, x2)), np.array(k.grad(x2, x1)).swapaxes(1, 2))
    nt.assert_allclose(k.get(x1), k.get(x1, x1))
    nt.assert_allclose(np.array(k.dgrad(x1)), [np.diag(_) for _ in k.grad(x1)])
    h = k.get_hyper()
    f = lambda h_, a, b: k.copy_with(h_).get(a[None], b[None])[0, 0]
    G2 = np.array([spop.approx_fprime(h, f, 1e-8, a, b) for a in x1 for b in x2])
    G2 = G2.swapaxes(0, 1).reshape(-1, x1.shape[0], x2.shape[0])
    nt.assert_allclose(np.array(k.grad(x1, x2)), G2, rtol=1e-6, atol=1e-6)


def _build(name):
    spec, N, d, fitc = GP_CASES[name]
    X, y, Xs, U = gp_inputs(N, d, fitc)
    k = make_kernel(spec)
    gp = OFITC(GP_SN, k, GP_MEAN, U) if fitc else OExactGP(GP_SN, k, GP_MEAN)
    gp.add_data(X, y)
    return gp, Xs


@pytest.mark.parametrize('name', sorted(GP_CASES))
def test_gp_vs_golden(name, golden):
    g = golden['gp']
    gp, Xs = _build(name)
    lZ, dlZ = gp.loglikelihood(True)
    mu, s2, dmu, ds2 = gp.posterior(Xs, grad=True)
    nt.assert_allclose(dmu, g[name + '/dmu'], rtol=1e-10, atol=1e-12)
    nt.assert_allclose(ds2, g[name + '/ds2'], rtol=1e-10, atol=1e-12)
    fmu, fS = gp.full_posterior(g[name + '/Xj'])
    nt.assert_allclose(fmu, g[name + '/full_mu'], rtol=1e-12)
    nt.assert_allclose(fS, g[name + '/full_Sigma'], rtol=1e-10, atol=1e-13)
    nt.assert_allclose(gp.sample(g[name + '/Xj'], 3, latent=False, rng=5), g[name + '/sample'], rtol=1e-8, atol=1e-9)
    nt.assert_allclose(lZ, g[name + '/lZ'], rtol=1e-12)
    nt.assert_allclose(dlZ, g[name + '/dlZ'], rtol=1e-10, atol=1e-10)
    nt.assert_allclose(mu, g[name + '/mu'], rtol=1e-12)
    nt.assert_allclose(s2, g[name + '/s2'], rtol=1e-10, atol=1e-14)
    gp.set_hyper(g[name + '/hyper2'])
    lZ, dlZ = gp.loglikelihood(True)
    nt.assert_allclose(lZ, g[name + '/lZ_h2'], rtol=1e-12)
    nt.assert_allclose(dlZ, g[name + '/dlZ_h2'], rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize('name', sorted(SURVEY_KAT))
def test_gp_vs_survey_kat(name):
    lZ0, dlZ0, mu0, s20 = SURVEY_KAT[name]
    gp, Xs = _build(name)
    lZ, dlZ = gp.loglikelihood(True)
    mu, s2 = gp.posterior(Xs)
    nt.assert_allclose(lZ, lZ0, rtol=1e-10)
    nt.assert_allclose(dlZ, dlZ0, rtol=1e-8, atol=1e-9)
    nt.assert_allclose(mu, mu0, rtol=1e-10)
    nt.assert_allclose(s2, s20, rtol=1e-9)


@pytest.mark.parametrize('name', ['se_ard_3d', 'fitc_se_2d'])
def test_gp_grad_fd(name):
    # tests/test_inference.py:105-112
    gp, _ = _build(name)
    import copy
    h = gp.get_hyper()

    def f(h_):
        g2 = copy.deepcopy(gp)
        g2.set_hyper(h_)
        return g2.loglikelihood()
    _, g1 = gp.loglikelihood(True)
    nt.assert_allclose(g1, spop.approx_fprime(h, f, 1e-8), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize('name', sorted(GP_CASES) + sorted(DTC_CASES))
def test_reference_record(name, golden):
    """The reference outputs in tests/golden that the other golden tests leave unchecked: the
    hyper layout, the exact-GP factor R and whitened residual a, and the outputs after
    set_hyper(hyper2), at the tolerances oracle/make_golden.py compared them with when it
    recorded them (its default 1e-12 / 1e-13 for R, a and the exact/FITC posterior after
    set_hyper, which it stored unchecked).  With them every stored reference array is compared."""
    from oracle.pygp_oracle import ODTC
    g = golden['gp']
    if name in DTC_CASES:
        spec, N, d = DTC_CASES[name]
        X, y, Xs, U = gp_inputs(N, d, True)
        gp = ODTC(GP_SN, make_kernel(spec), GP_MEAN, U)
        gp.add_data(X, y)
        nt.assert_allclose(gp.full_posterior(Xs)[1], g[name + '/full_Sigma'], rtol=1e-8, atol=1e-11)
        gp.set_hyper(g[name + '/hyper2'])
        lZ, dlZ = gp.loglikelihood(True)
        mu, s2, dmu, ds2 = gp.posterior(Xs, grad=True)
        nt.assert_allclose(lZ, g[name + '/lZ_h2'], rtol=1e-12)
        nt.assert_allclose(dlZ, g[name + '/dlZ_h2'], rtol=1e-9, atol=1e-10)
        nt.assert_allclose(mu, g[name + '/mu_h2'], rtol=1e-10, atol=1e-12)
        nt.assert_allclose(s2, g[name + '/s2_h2'], rtol=1e-9, atol=1e-12)
        nt.assert_allclose(dmu, g[name + '/dmu_h2'], rtol=1e-9, atol=1e-11)
        nt.assert_allclose(ds2, g[name + '/ds2_h2'], rtol=1e-8, atol=1e-11)
        nt.assert_allclose(gp.full_posterior(Xs)[1], g[name + '/full_Sigma_h2'], rtol=1e-8, atol=1e-11)
        return
    gp, Xs = _build(name)
    nt.assert_array_equal(gp.get_hyper(), g[name + '/hyper'])
    if not GP_CASES[name][3]:
        R = g[name + '/R']
        nt.assert_allclose(gp._R[:R.shape[0], :R.shape[1]], R, rtol=1e-12, atol=1e-13)
        nt.assert_allclose(gp._a, g[name + '/a'], rtol=1e-12, atol=1e-13)
    gp.set_hyper(g[name + '/hyper2'])
    mu, s2 = gp.posterior(Xs)
    nt.assert_allclose(mu, g[name + '/mu_h2'], rtol=1e-12, atol=1e-13)
    nt.assert_allclose(s2, g[name + '/s2_h2'], rtol=1e-11, atol=1e-13)


@pytest.mark.parametrize('name', ['fitc_se_2d', 'fitc_ard4_500'])
def test_fitc_device_model(name):
    """The regrouped FITC algebra the device runs (oracle/fitc_model.py: transposed
    layout, gradient as three elementwise traces) equals fitc.py's own loop."""
    from oracle import fitc_model as fm
    spec, N, d, _ = GP_CASES[name]
    X, y, Xs, U = gp_inputs(N, d, True)
    k = make_kernel(spec)
    gp = OFITC(GP_SN, k, GP_MEAN, U)
    gp.add_data(X, y)
    lZ, dlZ = gp.loglikelihood(True)
    mu, s2 = gp.posterior(Xs)
    st = fm.fitc_update(k, GP_SN**2, GP_MEAN, U, X, y)
    lZ2, dlZ2 = fm.fitc_loglike(k, st, U, X, True)
    mu2, s22 = fm.fitc_predict(k, st, U, Xs)
    nt.assert_allclose(lZ2, lZ, rtol=1e-11)
    nt.assert_allclose(dlZ2, dlZ, rtol=1e-9, atol=1e-9*np.abs(dlZ).max())
    nt.assert_allclose(mu2, mu, rtol=1e-11, atol=1e-12)
    nt.assert_allclose(s22, s2, rtol=1e-10, atol=1e-13)


@pytest.mark.parametrize('N', [63, 64, 129, 257, 700])
def test_exact_device_model(N):
    """The blocked formulation the device runs (oracle/blocked_model.py: recursive
    right-looking Cholesky with r riding along, bottom-up triangular inverse,
    lower-triangle trace) reaches the parity bars against the oracle."""
    from oracle import blocked_model as bm
    from oracle.pygp_oracle import synthetic_problem
    X, y, Xs = synthetic_problem(N, 3, 9)
    spec = ('matern', 1.0, [0.5, 0.6, 0.7], 5)
    gp = OExactGP(0.1, make_kernel(spec), 0.2)
    gp.add_data(X, y)
    lZ, dlZ = gp.loglikelihood(True)
    mu, s2 = gp.posterior(Xs)
    out = bm.device_model(make_kernel(spec), 0.1, 0.2, X, y, True, Xs)
    assert out['info'] == 0
    nt.assert_allclose(out['lZ'], lZ, rtol=1e-11)
    nt.assert_allclose(out['dlZ'], dlZ, rtol=1e-9, atol=1e-9*np.abs(dlZ).max())
    nt.assert_allclose(out['mu'], mu, rtol=1e-10, atol=1e-11)
    nt.assert_allclose(out['s2'], s2, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize('name', ['dtc_se_2d', 'dtc_ard4_500'])
def test_dtc_vs_golden_and_device_model(name, golden):
    """ODTC against the reference's outputs, and the regrouped DTC algebra the device
    runs (oracle/fitc_model.py: dtc_*) against ODTC."""
    from oracle import fitc_model as fm
    from oracle.cases import DTC_CASES
    from oracle.pygp_oracle import ODTC
    g = golden['gp']
    spec, N, d = DTC_CASES[name]
    X, y, Xs, U = gp_inputs(N, d, True)
    k = make_kernel(spec)
    gp = ODTC(GP_SN, k, GP_MEAN, U)
    gp.add_data(X, y)
    lZ, dlZ = gp.loglikelihood(True)
    mu, s2, dmu, ds2 = gp.posterior(Xs, grad=True)
    nt.assert_allclose(lZ, g[name + '/lZ'], rtol=1e-12)
    nt.assert_allclose(dlZ, g[name + '/dlZ'], rtol=1e-9, atol=1e-10)
    nt.assert_allclose(mu, g[name + '/mu'], rtol=1e-10, atol=1e-12)
    nt.assert_allclose(s2, g[name + '/s2'], rtol=1e-9, atol=1e-12)
    nt.assert_allclose(dmu, g[name + '/dmu'], rtol=1e-9, atol=1e-11)
    nt.assert_allclose(ds2, g[name + '/ds2'], rtol=1e-8, atol=1e-11)
    st = fm.dtc_update(k, GP_SN**2, GP_MEAN, U, X, y)
    lZ2, dlZ2 = fm.dtc_loglike(k, st, U, X, True)
    mu2, s22 = fm.dtc_predict(k, st, U, Xs)
    nt.assert_allclose(lZ2, lZ, rtol=1e-11)
    nt.assert_allclose(dlZ2, dlZ, rtol=1e-9, atol=1e-9*np.abs(dlZ).max())
    nt.assert_allclose(mu2, mu, rtol=1e-10, atol=1e-11)
    nt.assert_allclose(s22, s2, rtol=1e-10, atol=1e-13)
