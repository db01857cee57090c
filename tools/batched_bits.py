"""Seeded outputs of the batched exact-GP path, for bitwise comparison between two builds:
pgp_batched_loglike without and with dlZ and pgp_batched_predict, for an SE-ARD, a Matern-5/2, an
SE+Periodic and an RQ kernel, B = 1 and 6.

    python tools/batched_bits.py dump TREE OUT.npz     # with TREE's build of the package
    python tools/batched_bits.py compare A.npz B.npz   # exit 1 unless every array is bitwise equal
"""

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = [   # spec, n, d, ms, name
    (('se', 1.0, [0.5]*8), 2048, 8, 37, 'se8'),
    (('matern', 1.0, [0.6]*3, 5), 3001, 3, 129, 'm5'),
    (('sum', ('se', 1.0, 0.5), ('periodic', 0.5, 1.0, 0.25)), 700, 1, 64, 'sp'),
    (('rq', 0.5, [0.4, 0.5], 0.3), 100, 2, 5, 'rq'),
]


def dump(tree, path):
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    sys.path.insert(0, os.path.abspath(tree))
    import pygp_b200 as pygp
    from pygp_b200 import sharding
    from gpu_util import product_kernel
    res = {}
    for spec, n, d, ms, name in CASES:
        rng = np.random.RandomState(n)
        X, Xs = rng.rand(n, d), rng.rand(ms, d)
        y = np.sin(3*X.sum(1)) + 0.1*rng.randn(n)
        gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), product_kernel(spec), 0.0)
        gp.add_data(X, y)
        for B in (1, 6):
            H = gp.get_hyper() + rng.uniform(-0.2, 0.2, size=(B, gp.nhyper))
            res['%s_%d_lZ' % (name, B)] = sharding._batched('loglike', gp, H, None)
            res['%s_%d_lZg' % (name, B)] = sharding._batched('loglike_grad', gp, H, None)
            res['%s_%d_mu' % (name, B)], res['%s_%d_s2' % (name, B)] = sharding._batched('predict', gp, H, Xs)
    np.savez(path, **res)
    print('%s: %d arrays from %s' % (path, len(res), os.path.abspath(tree)))


def compare(pa, pb):
    a, b = np.load(pa), np.load(pb)
    bad = sorted(k for k in set(a.files) | set(b.files)
                 if k not in a.files or k not in b.files or not np.array_equal(a[k], b[k], equal_nan=True))
    print('bitwise: %d arrays, %d differ %s' % (len(a.files), len(bad), bad))
    return 1 if bad else 0


if __name__ == '__main__':
    if len(sys.argv) == 4 and sys.argv[1] == 'dump':
        dump(sys.argv[2], sys.argv[3])
    elif len(sys.argv) == 4 and sys.argv[1] == 'compare':
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
