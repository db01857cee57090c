"""
Type-II maximum likelihood (pygp/learning/optimization.py:21-67).

The optimiser (scipy L-BFGS-B) stays on the host; each objective evaluation is
`set_hyper` + `loglikelihood(True)`, i.e. one pgp_exact_update and one
pgp_exact_loglike on data that never leaves HBM.  With `pseudoinputs=True` a
FITC / DTC model also fits its pseudo-inputs: each evaluation moves U without
re-factorising, then `set_hyper` factorises once and
`loglikelihood(True, pseudoinputs=True)` returns the gradient in U as well.
"""

import numpy as np
import scipy.optimize as so

from ..utils.models import get_params

__all__ = ['optimize']


def optimize(gp, priors=None, pseudoinputs=False):
    """Fit the hypers of `gp` in place.  `priors` maps parameter names to
    None (hold that block fixed); proper priors are unsupported, as in the
    reference (optimization.py:50-52).  `pseudoinputs=True` fits the
    pseudo-inputs of a sparse model (FITC, DTC) jointly with the active hypers."""
    if pseudoinputs and not hasattr(gp, 'pseudoinputs'):
        raise ValueError('pseudoinputs=True needs a model with pseudo-inputs (FITC, DTC)')
    hyper0 = gp.get_hyper()
    active = np.ones(gp.nhyper, dtype=bool)
    blocks = dict((name, block) for name, block, _ in get_params(gp))
    for name, prior in (priors or {}).items():
        if prior is not None:
            raise AssertionError('optimize only supports priors that fix a parameter (None)')
        active[blocks[name]] = False

    def objective(x):
        hyper = hyper0.copy()
        hyper[active] = x
        gp.set_hyper(hyper)
        lZ, dlZ = gp.loglikelihood(True)
        return -lZ, -dlZ[active]

    if not pseudoinputs:
        x, _, _ = so.fmin_l_bfgs_b(objective, hyper0[active])
        hyper = hyper0.copy()
        hyper[active] = x
        gp.set_hyper(hyper)
        return

    shape, na = gp.pseudoinputs.shape, int(active.sum())

    def objective_u(x):
        hyper = hyper0.copy()
        hyper[active] = x[:na]
        gp._set_pseudoinputs(x[na:].reshape(shape))
        gp.set_hyper(hyper)
        lZ, dlZ, dU = gp.loglikelihood(True, pseudoinputs=True)
        return -lZ, -np.r_[dlZ[active], dU.ravel()]

    x, _, _ = so.fmin_l_bfgs_b(objective_u, np.r_[hyper0[active], gp.pseudoinputs.ravel()])
    hyper = hyper0.copy()
    hyper[active] = x[:na]
    gp._set_pseudoinputs(x[na:].reshape(shape))
    gp.set_hyper(hyper)
