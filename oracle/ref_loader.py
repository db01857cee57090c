"""
TEST INFRASTRUCTURE ONLY -- import the UNMODIFIED reference (Python-2 era
mwhoffman/pygp; PYGP_REFERENCE_ROOT names a source checkout of it).

Nothing in that checkout is edited or copied; the py2-isms are bridged at
run time (SURVEY.md section 8c).  The reference is not part of this
repository, so only ``oracle/make_golden.py`` uses this module: it records the
reference's outputs under tests/golden, which the tests compare against.
"""

import builtins
import itertools
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get('PYGP_REFERENCE_ROOT', '/root/reference')


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'pygp'))


def _install_mwhutils():
    """Stand-in for the un-vendored third-party `mwhutils` (requirements.txt:4
    pins it to a git URL with no version): only the four entry points pygp
    imports.  `chol_update` restates the textbook block update
    R' = [[R, S],[0, chol(Kss - S^T S)]], S = R^-T Kxs, a' = [a, R22^-T(r - S^T a)]."""
    import abc as _abc
    import scipy.linalg as sla

    root = types.ModuleType('mwhutils')
    m_abc = types.ModuleType('mwhutils.abc')
    m_abc.ABCMeta = _abc.ABCMeta
    m_abc.abstractmethod = _abc.abstractmethod

    class abstractclassmethod(classmethod):
        __isabstractmethod__ = True

        def __init__(self, f):
            f.__isabstractmethod__ = True
            super(abstractclassmethod, self).__init__(f)
    m_abc.abstractclassmethod = abstractclassmethod

    m_random = types.ModuleType('mwhutils.random')

    def rstate(rng=None):
        if rng is None:
            return np.random.mtrand._rand
        if isinstance(rng, np.random.RandomState):
            return rng
        return np.random.RandomState(rng)

    def grid(bounds, n):
        bounds = np.array(bounds, ndmin=2, dtype=float)
        axes = [np.linspace(a, b, n) for a, b in bounds]
        return np.stack(np.meshgrid(*axes, indexing='ij'), -1).reshape(-1, len(axes))
    m_random.rstate = rstate
    m_random.grid = grid

    m_linalg = types.ModuleType('mwhutils.linalg')

    def chol_update(R, Kxs, Kss, a, r):
        S = sla.solve_triangular(R, Kxs, trans=True)
        R22 = sla.cholesky(Kss - S.T.dot(S))
        n, m = R.shape[0], R22.shape[0]
        Rn = np.zeros((n+m, n+m))
        Rn[:n, :n], Rn[:n, n:], Rn[n:, n:] = R, S, R22
        an = np.r_[a, sla.solve_triangular(R22, r - S.T.dot(a), trans=True)]
        return Rn, an
    m_linalg.chol_update = chol_update

    root.abc, root.random, root.linalg = m_abc, m_random, m_linalg
    sys.modules.update({'mwhutils': root, 'mwhutils.abc': m_abc,
                        'mwhutils.random': m_random,
                        'mwhutils.linalg': m_linalg})


def load():
    """Return the reference `pygp` package, imported from REFERENCE_ROOT."""
    if 'pygp' in sys.modules and getattr(sys.modules['pygp'], '_is_reference', False):
        return sys.modules['pygp']
    if not available():
        raise ImportError('reference tree not present at %s' % REFERENCE_ROOT)

    # shim 1/2: py2 builtins used by the reference.
    builtins.xrange = range
    itertools.izip = zip
    # shim 3: scipy.misc.logsumexp (meta/smc.py:13).
    import scipy.special
    misc = types.ModuleType('scipy.misc')
    misc.logsumexp = scipy.special.logsumexp
    sys.modules['scipy.misc'] = misc
    # shim 4: mwhutils stand-in.
    _install_mwhutils()
    # shim 5: np.hstack/np.vstack fed generators (_combo.py:91, priors.py:91).
    _hstack, _vstack = np.hstack, np.vstack

    def hstack(tup, *a, **k):
        return _hstack(list(tup) if not isinstance(tup, (list, tuple, np.ndarray)) else tup, *a, **k)

    def vstack(tup, *a, **k):
        return _vstack(list(tup) if not isinstance(tup, (list, tuple, np.ndarray)) else tup, *a, **k)
    np.hstack, np.vstack = hstack, vstack
    # shim 6: matplotlib stub (demos import pyplot).
    if 'matplotlib' not in sys.modules:
        mpl = types.ModuleType('matplotlib')
        plt = types.ModuleType('matplotlib.pyplot')
        mpl.pyplot = plt
        sys.modules['matplotlib'] = mpl
        sys.modules['matplotlib.pyplot'] = plt

    sys.path.insert(0, REFERENCE_ROOT)
    try:
        import pygp
    finally:
        sys.path.remove(REFERENCE_ROOT)
    import pygp.meta.mcmc as _mcmc
    _mcmc.map = lambda f, *a: list(map(f, *a))       # mcmc.py:76-79 subscripts a map
    pygp._is_reference = True
    return pygp


def ref_kernel(pygp, spec):
    """Build a REFERENCE kernel object from an oracle spec tuple."""
    pk = pygp.kernels
    tag = spec[0]
    if tag == 'se':
        return pk.SE(*spec[1:])
    if tag == 'matern':
        return pk.Matern(*spec[1:])
    if tag == 'periodic':
        return pk.Periodic(*spec[1:])
    if tag == 'rq':
        return pk.RQ(*spec[1:])
    parts = [ref_kernel(pygp, s) for s in spec[1:]]
    out = parts[0]
    for p in parts[1:]:
        out = (out + p) if tag == 'sum' else (out * p)
    return out
