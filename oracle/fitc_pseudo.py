"""
TEST INFRASTRUCTURE ONLY -- a numpy model of the pseudo-input gradient of the
FITC / DTC log marginal likelihood in the device formulation
(pygp_b200/csrc/fitc.cu pgp_fitc_loglike_pseudo, gram.cu pseudo_gram_kernel),
built from the intermediates of oracle/fitc_model.py.

The regrouped hyper-gradient of fitc_model.py,

  dlZ_h = 1/2 [ dk_h(0) sum(q - 1/ell^2) + sum(dKuu_h o Cuu) + sum(dKxu_h o Cxu) ],

holds for any parameter Kuu, Kxu and kxx depend on.  For a pseudo-input
coordinate u_jk of a stationary kernel, d kxx / d u = 0 and d k(u, u) / d u = 0,
and the su2 jitter does not depend on U, so with Cuu symmetric

  dlZ / dU[j, k] =      sum_i Cuu[j, i] d k(u_j, u_i) / d u_jk      (i < p)
                 + sx * sum_i Cxu[i, j] d k(u_j, x_i) / d u_jk      (i < n)

with sx = 1/2 (FITC) or 1 / (2 sqrt(sn2)) (DTC, whose Cxu has q = 1).
tests/test_fitc_pseudoinputs.py checks this against central differences of
the oracle's lZ in every entry of U.
"""

import numpy as np
import scipy.linalg as sla


def _contract(kernel, U, X, Cuu, Cxu, sx):
    Guu = kernel.gradx(U, U)        # (p, p, d): d k(u_j, u_i) / d u_j
    Gux = kernel.gradx(U, X)        # (p, n, d): d k(u_j, x_i) / d u_j
    return np.einsum('ji,jik->jk', Cuu, Guu) + sx*np.einsum('ij,jik->jk', Cxu, Gux)


def fitc_pseudo_grad(kernel, st, U, X):
    """dlZ / dU (p, d) of FITC from the state of fitc_model.fitc_update."""
    Lc, Al, Vs, ell, rs = st['Lc'], st['Al'], st['Vs'], st['ell'], st['rs']
    beta = sla.solve_triangular(Al, Vs.T.dot(rs), lower=True)
    t = sla.solve_triangular(Al, beta, lower=True, trans=1)
    alpha = (rs - Vs.dot(t)) / ell
    G = sla.solve_triangular(Lc, np.eye(len(Lc)), lower=True).T
    Bt = (Vs*ell[:, None]).dot(G.T)
    Wt = sla.solve_triangular(Al, (Vs/ell[:, None]).T, lower=True).T
    w = Bt.T.dot(alpha)
    q = alpha**2 + np.sum(Wt**2, axis=1)
    P = Bt.T.dot(Wt)
    Cuu = Bt.T.dot(Bt*q[:, None]) - P.dot(P.T) - np.outer(w, w)
    Cxu = 2*(np.outer(alpha, w) - Bt*q[:, None] + Wt.dot(P.T))
    return _contract(kernel, U, X, Cuu, Cxu, 0.5)


def dtc_pseudo_grad(kernel, st, U, X):
    """dlZ / dU (p, d) of DTC from the state of fitc_model.dtc_update."""
    Luu, Al, Vs, rs, beta, ell = st['Luu'], st['Al'], st['Vs'], st['rs'], st['beta'], st['ell']
    alpha = rs - Vs.dot(sla.solve_triangular(Al, beta, lower=True, trans=1))
    Bt = sla.solve_triangular(Luu, Vs.T, lower=True, trans=1).T
    Wt = sla.solve_triangular(Al, Vs.T, lower=True).T
    w = Bt.T.dot(alpha)
    P = Bt.T.dot(Wt)
    Cuu = Bt.T.dot(Bt) - P.dot(P.T) - np.outer(w, w)
    Cxu = 2*(np.outer(alpha, w) - Bt + Wt.dot(P.T))
    return _contract(kernel, U, X, Cuu, Cxu, 0.5/ell)
