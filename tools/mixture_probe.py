"""Mixture posterior with input-gradients (meta.MCMC.posterior(X, grad=True)) on the
GPU: the per-model loop over materialised ExactGP copies against the resident
batch (pgp_batch + xgrad_gram_kernel), alternating, and the contraction kernel's
rate beside the mode-2 Gram kernel's.  Writes profiles/r05_mixture_grad.txt
(or the path given as the first argument).

    python tools/mixture_probe.py [out.txt]
"""

import gc
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pygp_b200 as pygp                               # noqa: E402
from pygp_b200 import _lib                             # noqa: E402
from pygp_b200.meta.mcmc import _DeviceBatch, _mixture  # noqa: E402

PC_GRAM = 1
D, B, RUNS = 8, 100, 3
LINES = []


def out(s):
    print(s, flush=True)
    LINES.append(s)


def card():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    return subprocess.check_output(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader']).decode().strip()


def problem(n, ms, seed=0):
    rng = np.random.RandomState(seed)
    X, Xs = rng.rand(n, D), rng.rand(ms, D)
    y = np.sin(3*X.sum(1)) + 0.1*rng.randn(n)
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [0.5]*D), 0.0)
    gp.add_data(X, y)
    H = gp.get_hyper() + rng.uniform(-0.2, 0.2, size=(B, gp.nhyper))
    return gp, H, Xs


def timed(fn):
    ctx = _lib.context()
    ctx.sync()
    t0 = time.perf_counter()
    r = fn()
    ctx.sync()
    return time.perf_counter() - t0, r


def loop_first(gp, H, Xs):
    models = [gp.copy(h) for h in H]                          # the parent's MCMC._samples
    parts = [m.posterior(Xs, True) for m in models]
    return models, _mixture(*(np.array([p[i] for p in parts]) for i in range(4)))


def loop_steady(models, Xs):
    parts = [m.posterior(Xs, True) for m in models]
    return _mixture(*(np.array([p[i] for p in parts]) for i in range(4)))


def batch_first(gp, H, Xs, budget=0):
    bt = _DeviceBatch(gp, H, budget)
    return bt, _mixture(*bt.predict(Xs, True))


def compare(n, ms):
    gp, H, Xs = problem(n, ms)
    res = {'loop_first': [], 'loop_steady': [], 'batch_first': [], 'batch_steady': []}
    diff = 0.0
    for r in range(RUNS + 1):               # run 0 warms every shape up and is not reported
        t1, (models, ref) = timed(lambda: loop_first(gp, H, Xs))
        t2, _ = timed(lambda: loop_steady(models, Xs))
        del models
        gc.collect()
        t3, (bt, got) = timed(lambda: batch_first(gp, H, Xs))
        t4, _ = timed(lambda: _mixture(*bt.predict(Xs, True)))
        del bt
        gc.collect()
        if r:
            for k, t in zip(res, (t1, t2, t3, t4)):
                res[k].append(t)
        for a, b in zip(got, ref):
            diff = max(diff, float(np.abs(a - b).max() / max(1.0, np.abs(b).max())))
    med = {k: float(np.median(v)) for k, v in res.items()}
    out('N=%5d ms=%3d  loop first %8.4f s steady %8.4f s | batch first %8.4f s steady %8.4f s | '
        'first x%.1f steady x%.1f | runs loop %s batch %s | max rel diff %.1e'
        % (n, ms, med['loop_first'], med['loop_steady'], med['batch_first'], med['batch_steady'],
           med['loop_first']/med['batch_first'], med['loop_steady']/med['batch_steady'],
           ['%.4f' % t for t in res['loop_steady']], ['%.4f' % t for t in res['batch_steady']], diff))


def kernel_rates(n=8192):
    ctx = _lib.context()
    for ms in (1, 256):
        gp, H, Xs = problem(n, ms)
        bt = _DeviceBatch(gp, H)
        bt.predict(Xs, True)
        bt.predict(Xs)
        ctx.profile(True)
        bt.predict(Xs)
        _, t_plain, _ = ctx.profile_read(PC_GRAM)
        ctx.profile(True)
        bt.predict(Xs, True)
        nl, t_grad, _ = ctx.profile_read(PC_GRAM)
        ctx.profile(False)
        t_x = t_grad - t_plain                                   # the contraction kernel's launches
        steady = float(np.median([timed(lambda: bt.predict(Xs, True))[0] for _ in range(RUNS)]))
        entries = float(B) * ms * n * D
        out('xgrad_gram_kernel N=%d ms=%d d=%d B=%d: %.3f ms, %.3e gradient entries/s, %.1f %% of the %.2f ms '
            'steady pgp_batch_predict call (PC_GRAM %d launches, k(X*, X) Gram %.3f ms)'
            % (n, ms, D, B, t_x, entries / (t_x * 1e-3), 100.0 * t_x * 1e-3 / steady, steady * 1e3, nl, t_plain))
        del bt
        gc.collect()
    # mode-2 gram_kernel (d k / d x1[k], written to memory), at a size that fills the GPU: 2048 x 8192 entries per
    # launch (4096 CTAs), one launch per dimension
    n1 = 2048
    rng = np.random.RandomState(1)
    X1, X2 = rng.rand(n1, D), rng.rand(n, D)
    k = pygp.kernels.SE(1.0, [0.5]*D)
    k.gradx(X1, X2)
    ctx.profile(True)
    k.gradx(X1, X2)
    nl, t_g, _ = ctx.profile_read(PC_GRAM)
    ctx.profile(False)
    e2 = float(n1) * n * D
    out('gram_kernel mode 2 (gradx, entries written to HBM) n1=%d n2=%d d=%d: %.3f ms in %d launches, %.3e entries/s'
        % (n1, n, D, t_g, nl, e2 / (t_g * 1e-3)))


def large(n=16384, ms=256):
    gp, H, Xs = problem(n, ms)
    per = 8*((n + 1)*((n + 15)//16*16) + ((n + 63)//64*64 + 64)*D + 1) + 8192
    for label, budget in (('default budget', 0), ('budget of 67 factors', 67*per)):
        t1, (bt, _) = timed(lambda: batch_first(gp, H, Xs, budget))
        ts = []
        for _ in range(RUNS):
            t, _ = timed(lambda: _mixture(*bt.predict(Xs, True)))
            ts.append(t)
        out('N=%d ms=%d B=%d %s: resident %d of %d, first %.3f s, steady %s s'
            % (n, ms, B, label, bt.resident, B, t1, ['%.3f' % t for t in ts]))
        del bt
        gc.collect()
    out('N=%d loop: not measured (%d factors of %.1f GB do not fit the card)' % (n, B, 8.0*n*n/1e9))


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles', 'r05_mixture_grad.txt')
    out('# tools/mixture_probe.py: MCMC.posterior(X, grad=True), SE-ARD d=%d, B=%d; medians of %d runs, '
        'loop (parent: one ExactGP copy per sample) and batch (pgp_batch) alternating' % (D, B, RUNS))
    out('# card (name, power limit, SM clock, max SM clock): ' + card())
    for n in (512, 2048, 8192):
        for ms in (1, 256):
            compare(n, ms)
    kernel_rates()
    large()
    out('# card after: ' + card())
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as f:
        f.write('\n'.join(LINES) + '\n')


if __name__ == '__main__':
    main()
