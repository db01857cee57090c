"""The emulated-FP64 V V^T of the exact-GP gradient (pygp_b200/csrc/ozaki.cu), checked through
tools/bin/ozaki_check: the INT8 residue products bit-exact, the reconstruction against exact Python
integers (entries that cancel heavily, trap 1), the residues of int64 values above 2^53 (trap 2), the
emulated product against the DMMA one on a real Matern-5/2 factor, and the gradient end to end."""

import json
import os
import subprocess

import numpy as np
import pytest

from gpu_util import assert_grad_close, LZ_RTOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECK = os.path.join(ROOT, 'tools', 'bin', 'ozaki_check')
MODULI = [256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193]
N_MIN = 8192          # chol.cu kOzakiMinN: the smallest order that takes the emulated product

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def check():
    import __graft_entry__ as g
    g.build()
    return CHECK


def run(*args):
    p = subprocess.run([CHECK] + [str(a) for a in args], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


@pytest.mark.parametrize('n', [1, 127, 129, 1000, 4100])
def test_residue_products_bit_exact(check, n):
    out = run('exact', n)
    assert 'residue_mismatches=0' in out and 'exponent_mismatches=0' in out and 'merge_over_4ulp=0' in out, out


def test_non_finite_rows_give_nan(check):
    assert 'wrong=0' in run('nonfinite', 0)


def ulps(a, b):
    if a == b:
        return 0.0
    return abs(a - b) / np.spacing(max(abs(a), abs(b)))


def test_reconstruction_of_cancelling_entries(check, tmp_path):
    path = tmp_path / 'merge.txt'
    run('merge', path)
    worst, count = 0.0, 0
    for line in open(path):
        xs, vs = line.split()
        x = int(xs)
        worst = max(worst, ulps(float(vs), float(x)))     # float(int) is correctly rounded
        count += 1
    assert count == 128 * 129 // 2
    assert worst <= 4, worst


def test_residues_above_2_53(check, tmp_path):
    path = tmp_path / 'resid.txt'
    run('resid', path)
    count = 0
    for line in open(path):
        f = [int(v) for v in line.split()]
        x, r = f[0], f[1:]
        assert abs(x) > 2**53
        for m, rt in zip(MODULI, r):
            assert -128 <= rt <= 127 and (rt - x) % m == 0, (x, m, rt)
        count += 1
    assert count > 4000


@pytest.mark.parametrize('n', [N_MIN, 32768])
def test_emulated_matches_dmma(check, n):
    rec = json.loads(run('compare', n, 1).strip().splitlines()[-1])
    assert rec['max_rel_dH'] <= 1e-13, rec


def test_exactgp_gradient_at_min_n(check):
    import pygp_b200 as pygp
    from oracle.pygp_oracle import make_kernel, OExactGP, synthetic_problem
    n, d = N_MIN, 3
    X, y, _ = synthetic_problem(n, d, 0, seed=5)
    ell = [0.5 * np.sqrt(d)] * d
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), pygp.kernels.Matern(1.0, ell, 5), 0.0)
    gp.add_data(X, y)
    lZ, dlZ = gp.loglikelihood(True)
    ogp = OExactGP(0.1, make_kernel(('matern', 1.0, ell, 5)), 0.0)
    ogp.add_data(X, y)
    olZ, odlZ = ogp.loglikelihood(True)
    np.testing.assert_allclose(lZ, olZ, rtol=LZ_RTOL)
    assert_grad_close(dlZ, odlZ)


def test_batched_gradient_at_min_n_matches_single_model(check):
    """The batched gradient runs its problems on several streams and keeps the DMMA product; the
    single-model gradient takes the emulated one from N_MIN on.  Both must agree."""
    import ctypes as C
    import pygp_b200 as pygp
    from pygp_b200 import _lib
    from oracle.pygp_oracle import synthetic_problem
    n, d, B = N_MIN, 3, 3
    X, y, _ = synthetic_problem(n, d, 0, seed=6)
    k = pygp.kernels.Matern(1.0, [0.5 * np.sqrt(d)] * d, 5)
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), k, 0.0)
    gp.add_data(X, y)
    h0 = gp.get_hyper()
    H = h0 + np.random.RandomState(3).uniform(-0.3, 0.3, (B, len(h0)))
    lZ, dlZ, info = np.empty(B), np.empty((B, len(h0))), np.zeros(B, dtype=np.int32)
    ctx = _lib.context()
    _lib.check(ctx, _lib.lib().pgp_batched_loglike(ctx.handle, k._spec(), _lib.ptr(X), _lib.ptr(y), n,
                                                   _lib.ptr(H), B, _lib.ptr(lZ), _lib.ptr(dlZ),
                                                   info.ctypes.data_as(C.POINTER(C.c_int32))))
    assert not info.any()
    for b in range(B):
        gp.set_hyper(H[b])
        l1, g1 = gp.loglikelihood(True)
        np.testing.assert_allclose(lZ[b], l1, rtol=LZ_RTOL)     # the batched factorisation differs in the last bits
        np.testing.assert_allclose(dlZ[b], g1, rtol=1e-10, atol=1e-10 * np.abs(g1).max())
