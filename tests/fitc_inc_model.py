"""
TEST INFRASTRUCTURE ONLY -- a numpy model of the incremental FITC / DTC update
the device runs (pgp_fitc_append_inc, pygp_b200/csrc/fitc.cu, and
chol_update_lower, pygp_b200/csrc/chol.cu), in the device formulation of
oracle/fitc_model.py.  It runs the same Householder reflector sequence as the
kernel, so the algebra (which rows ride along, with which coefficients) is
checked against the oracle on the CPU, and the difference between the model
after appends and the model refactored on all the data is the reordering
floor the GPU tolerances allow for.  FITC and DTC share one append
(`sparse_append`), as they share one device entry point.  It lives beside the
tests that use it rather than in oracle/: oracle/ holds the checker and the
models of earlier device formulations, and stays as it is.

State (rows = data points):
  L    Lc = chol(Kuu + su2 I)  (DTC: Luu)           unchanged by appends
  A    Al = chol(I + Vs^T Vs), beta = Al^-1 Vs^T rs  rank-m update, beta rides with c = rs_new
  R    FITC: Rl = Lc Al = chol(Kuu + su2 I + Kux diag(1/ell^2) Kxu), b = Rl^-1 Kux (r/ell^2)
       DTC:  Rux = chol(Kuu + su2 I + Kux Kxu / sn2), b = Rux^-1 Kux r
       rank-m update by W = Kxu_new / ell_new; b rides with c = rs_new (FITC) or
       sn2 rs_new = sqrt(sn2) r_new (DTC), so that W^T c = Kux_new (r_new / ell_new^2) resp. Kux_new r_new
  Vs, ell, rs (n)  new rows appended, old rows unchanged
  slog = sum log ell, srs = sum rs^2                carried for lZ
"""

import numpy as np
import scipy.linalg as sla

from oracle import fitc_model as fm


def chol_update(L, Z, W, C):
    """L' L'^T = L L^T + W^T W and Z'[r] = L'^-1 (L Z[r] + W^T C[:, r]).

    L (n, n) lower with a positive diagonal, Z (extra, n) riding rows, W (m, n),
    C (m, extra).  Column k: the reflector H (L_kk, x) = (nrm, 0), x = W[:, k],
    H = I - tau v~ v~^T with v~ = (alpha - nrm, x) / mu scaled by mu = 2^ilogb(max |x_i|)
    (xs = x / mu, s = |xs|^2, v0 = -mu s / (alpha + nrm), tau = 2 / (v0^2 + s)),
    applied to (L_jk, W[:, j]) for every later row j and to (Z[r, k], C[:, r]):
        q = v0 a + xs.w,  a' = a - tau q v0,  w' = w - tau q xs   (mu = 0: identity).
    """
    L, Z = np.array(L, dtype=float), np.array(Z, dtype=float, ndmin=2)
    W, C = np.array(W, dtype=float, ndmin=2), np.array(C, dtype=float, ndmin=2)
    n = L.shape[0]
    for k in range(n):
        alpha = L[k, k]
        ym = np.abs(W[:, k]).max()
        if ym == 0:
            continue
        e = int(np.frexp(ym)[1]) - 1                  # ilogb
        mu = np.ldexp(1.0, e)
        x = np.ldexp(W[:, k], -e)
        s = x.dot(x)
        ec = max(int(np.frexp(alpha)[1]) - 1, e)
        nrm = np.ldexp(np.sqrt(np.ldexp(alpha, -ec)**2 + np.ldexp(mu, -ec)**2*s), ec)
        v0 = -(mu*s)/(alpha + nrm)
        tau = 2.0/(v0*v0 + s)
        L[k, k] = nrm
        W[:, k] = 0.0
        t = tau*(v0*L[k+1:, k] + x.dot(W[:, k+1:]))
        W[:, k+1:] -= np.outer(x, t)
        L[k+1:, k] -= t*v0
        t = tau*(v0*Z[:, k] + x.dot(C))
        C -= np.outer(x, t)
        Z[:, k] -= t*v0
    return L, Z


def _state(dtc, L, A, beta, R, b, Vs, ell, rs, sn2, su2, mean):
    return dict(dtc=dtc, L=L, A=A, beta=beta, R=R, b=b, Vs=Vs, ell=ell, rs=rs, sn2=sn2, su2=su2, mean=mean,
                slog=np.sum(np.log(ell)), srs=rs.dot(rs), n=len(rs))


def sparse_update(kernel, sn2, mean, U, X, y, dtc=False):
    """The state of a full update (oracle/fitc_model.py fitc_update / dtc_update)."""
    if dtc:
        st = fm.dtc_update(kernel, sn2, mean, U, X, y)
        ell = np.full(len(X), st['ell'])
        return _state(True, st['Luu'], st['Al'], st['beta'], st['Lux'], st['a'], st['Vs'], ell, st['rs'],
                      sn2, st['su2'], mean)
    st = fm.fitc_update(kernel, sn2, mean, U, X, y)
    beta = sla.solve_triangular(st['Al'], st['Vs'].T.dot(st['rs']), lower=True)
    return _state(False, st['Lc'], st['Al'], beta, st['Rl'], st['b'], st['Vs'], st['ell'], st['rs'],
                  sn2, st['su2'], mean)


def sparse_append(kernel, st, U, Xn, yn):
    """The state after appending the rows (Xn, yn): O(m p^2), as pgp_fitc_append_inc."""
    Xn, yn = np.array(Xn, dtype=float, ndmin=2), np.array(yn, dtype=float, ndmin=1)
    sn2, dtc = st['sn2'], st['dtc']
    Kxu = kernel.get(Xn, U)
    Vt = sla.solve_triangular(st['L'], Kxu.T, lower=True).T
    if dtc:
        ell = np.full(len(Xn), np.sqrt(sn2))
    else:
        ell = np.sqrt(kernel.dget(Xn) + sn2 - np.sum(Vt**2, axis=1))
    Vs = Vt/ell[:, None]
    rs = (yn - st['mean'])/ell
    A, beta = chol_update(st['A'], st['beta'], Vs, rs[:, None])
    c2 = rs*ell*ell if dtc else rs
    R, b = chol_update(st['R'], st['b'], Kxu/ell[:, None], c2[:, None])
    out = dict(st)
    out.update(A=A, beta=beta[0], R=R, b=b[0], Vs=np.r_[st['Vs'], Vs], ell=np.r_[st['ell'], ell],
               rs=np.r_[st['rs'], rs], slog=st['slog'] + np.sum(np.log(ell)), srs=st['srs'] + rs.dot(rs),
               n=st['n'] + len(yn))
    return out


def sparse_lz(st):
    """lZ from the factor and the carried sums (fitc_lz_kernel)."""
    return (-np.sum(np.log(np.diag(st['A']))) - st['slog'] - 0.5*(st['srs'] - st['beta'].dot(st['beta']))
            - 0.5*st['n']*np.log(2*np.pi))


def sparse_predict(kernel, st, U, Xs):
    """Marginal posterior (fitc_predict_reduce_kernel): mu, s2."""
    Ksu = kernel.get(Xs, U)
    LKt = sla.solve_triangular(st['L'], Ksu.T, lower=True).T
    RKt = sla.solve_triangular(st['R'], Ksu.T, lower=True).T
    m = RKt.dot(st['b'])
    mu = st['mean'] + (m/st['sn2'] if st['dtc'] else m)
    s2 = kernel.dget(Xs) + (np.sum(RKt**2, axis=1) - np.sum(LKt**2, axis=1))
    return mu, s2
