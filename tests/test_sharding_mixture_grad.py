"""The input-gradient form of the sharded mixture posterior (pygp_b200/sharding.py
sharded_mixture_posterior(grad=True)) on CPU: gloo process groups of 2 and 3 ranks,
with a host function of the hyper rows standing in for the per-rank device call.
The two all-reduce rounds must give the single-rank moment-matching formula of
meta/mcmc.py."""

import os
import socket

import numpy as np
import numpy.testing as nt
import pytest


def _components(H, X):
    """Deterministic stand-in for one posterior per hyper row: (mu_, s2_, dmu_, ds2_)."""
    a = H[:, :1]
    b = H[:, 1:2]
    z = X @ np.arange(1.0, X.shape[1] + 1)
    mu_ = np.sin(a*z[None] + b)
    s2_ = 1.0 + np.cos(b*z[None])**2
    w = np.arange(1.0, X.shape[1] + 1)
    dmu_ = (a*np.cos(a*z[None] + b))[:, :, None]*w
    ds2_ = (-2*b*np.cos(b*z[None])*np.sin(b*z[None]))[:, :, None]*w
    return mu_, s2_, dmu_, ds2_


def _reference(H, X):
    mu_, s2_, dmu_, ds2_ = _components(H, X)
    mu = np.mean(mu_, axis=0)
    s2 = np.mean(s2_ + (mu_ - mu)**2, axis=0)
    dmu = np.mean(dmu_, axis=0)
    Dmu = dmu_ - dmu
    ds2 = np.mean(ds2_ + 2*mu_[:, :, None]*Dmu - 2*mu[None, :, None]*Dmu, axis=0)
    return mu, s2, dmu, ds2


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, size, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=size)
    try:
        from pygp_b200 import sharding
        rng = np.random.RandomState(3)
        H = rng.uniform(0.5, 1.5, size=(7, 4))          # 7 samples: ragged over 2 and 3 ranks
        X = rng.rand(5, 3)
        got = sharding.sharded_mixture_posterior(None, H, X, local_fn=_components, grad=True)
        ref = _reference(H, X)
        assert got[2].shape == (5, 3) and got[3].shape == (5, 3)
        for a, b in zip(got, ref):
            nt.assert_allclose(a, b, rtol=1e-12, atol=1e-14)
        # a rank without samples (2 samples over 3 ranks) still takes part in both rounds
        got = sharding.sharded_mixture_posterior(None, H[:2], X, local_fn=_components, grad=True)
        for a, b in zip(got, _reference(H[:2], X)):
            nt.assert_allclose(a, b, rtol=1e-12, atol=1e-14)

        # a failure on one rank surfaces on every rank before the rounds
        def bad(h, x):
            if rank == size - 1:
                raise np.linalg.LinAlgError('not positive definite (last rank only)')
            return _components(h, x)
        try:
            sharding.sharded_mixture_posterior(None, H, X, local_fn=bad, grad=True)
            raise AssertionError('expected LinAlgError on every rank')
        except np.linalg.LinAlgError:
            pass
        got = sharding.sharded_mixture_posterior(None, H, X, local_fn=_components, grad=True)
        nt.assert_allclose(got[0], ref[0], rtol=1e-12, atol=1e-14)
        q.put((rank, 'ok'))
    except Exception:      # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_world_size_one_gradient_formula():
    from pygp_b200 import sharding
    rng = np.random.RandomState(4)
    H, X = rng.uniform(0.5, 1.5, size=(6, 4)), rng.rand(4, 2)
    got = sharding.sharded_mixture_posterior(None, H, X, local_fn=_components, grad=True)
    for a, b in zip(got, _reference(H, X)):
        nt.assert_allclose(a, b, rtol=1e-13, atol=1e-15)


@pytest.mark.timeout(240)
@pytest.mark.parametrize('size', [2, 3])
def test_gloo_gradient_rounds(size):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, size, port, q)) for r in range(size)]
    for p in procs:
        p.start()
    res = [q.get(timeout=200) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    for rank, msg in res:
        assert msg == 'ok', 'rank %d:\n%s' % (rank, msg)
