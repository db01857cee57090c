"""Measure every BASELINE.json config at full size on ONE GPU (run on the GPU box):
  C1 SE 1-D N=1000 + 500 test points        C2 SE-ARD d=8 N=8192 under learning.optimize
  C3 -> bench.py                            C4 4096 hyper samples x N=2048 (batched)
  C5 SE+Periodic 1-D N=65536 exact; FITC M=2048, N=2^20 (c5_fitc_pseudo: with d lZ / d U)
Prints one JSON line per config (profiles/r01b_configs.jsonl).  Timing: wall clock
around synchronous C-ABI calls (every call ends with a stream synchronise)."""

import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pygp_b200 as pygp     # noqa: E402
from pygp_b200 import _lib   # noqa: E402


def problem(n, d, seed=0):
    rng = np.random.RandomState(seed)
    X = rng.rand(n, d)
    y = np.sin(3*X.sum(1)) + 0.1*rng.randn(n)
    return X, y


def best(fn, reps=3):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        out.append(time.perf_counter() - t0)
    return min(out), r


def say(**kw):
    print(json.dumps(kw), flush=True)


def c1():
    X, y = problem(1000, 1)
    Xs = np.random.RandomState(1).rand(500, 1)
    gp = pygp.BasicGP(0.1, 1.0, 0.1, 0.0, ndim=1)
    gp.add_data(X, y)
    h = gp.get_hyper()

    def ev():
        gp.set_hyper(h)
        return gp.loglikelihood(True)
    ev()
    t_ev, (lZ, _) = best(ev, 5)
    gp.posterior(Xs)
    t_pr, _ = best(lambda: gp.posterior(Xs), 5)
    say(config='C1', workload='SE iso d=1 N=1000: set_hyper + loglikelihood(True); posterior on 500 points',
        eval_ms=t_ev*1e3, evals_per_s=1/t_ev, predict_ms=t_pr*1e3, predict_points_per_s=500/t_pr, lZ=lZ,
        reference_cpu='0.063 + 0.132 s per evaluation, 27.8 k pts/s (SURVEY.md 6, 8 vCPU)')


def c2():
    n, d = 8192, 8
    X, y = problem(n, d)
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.3), pygp.kernels.SE(1.5, [1.0]*d), 0.0)
    gp.add_data(X, y)
    calls = [0]
    orig = gp.loglikelihood

    def counted(grad=False):
        calls[0] += 1
        return orig(grad)
    gp.loglikelihood = counted
    lZ0 = orig()
    t0 = time.perf_counter()
    pygp.optimize(gp)
    t = time.perf_counter() - t0
    say(config='C2', workload='SE-ARD d=8 N=8192: learning.optimize (L-BFGS-B; each evaluation = set_hyper + loglikelihood(True))',
        evaluations=calls[0], seconds=t, evals_per_s=calls[0]/t, eff_fp64_tflops=calls[0]*float(n)**3/t/1e12,
        lZ_start=lZ0, lZ_end=orig(), reference_cpu='40.3 s per evaluation = 0.025 evals/s (SURVEY.md 6, 8 vCPU)')


def c4():
    n, d, B = 2048, 8, 4096
    X, y = problem(n, d)
    kern = pygp.kernels.SE(1.0, [0.5*np.sqrt(d)]*d)
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), kern, 0.0)
    gp.add_data(X, y)
    base = gp.get_hyper()
    H = base + np.random.RandomState(2).uniform(-0.5, 0.5, size=(B, len(base)))
    from pygp_b200 import sharding
    sharding.sharded_batched_loglike(gp, H[:64])
    t, lZ = best(lambda: sharding.sharded_batched_loglike(gp, H), 3)
    # spot-check 3 samples against single-model evaluations
    err = 0.0
    for i in (0, 1000, 4095):
        gp.set_hyper(H[i])
        err = max(err, abs(gp.loglikelihood() - lZ[i])/abs(lZ[i]))
    say(config='C4', workload='4096 hyper samples x N=2048 SE-ARD d=8: batched Gram + Cholesky + solve + lZ',
        seconds=t, samples_per_s=B/t, eff_fp64_tflops_potrf=B*float(n)**3/3/t/1e12, finite=int(np.isfinite(lZ).sum()),
        max_rel_err_vs_single=err)


def c5_exact():
    n = 65536
    rng = np.random.RandomState(0)
    X = np.sort(rng.rand(n, 1), axis=0)*64
    y = np.sin(3*X.sum(1)) + 0.1*rng.randn(n)
    k = pygp.kernels.SE(1.0, 0.5, ndim=1) + pygp.kernels.Periodic(0.5, 1.0, 0.25)
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), k, 0.0)
    t0 = time.perf_counter()
    gp.add_data(X, y)
    t_first = time.perf_counter() - t0
    h = gp.get_hyper()
    t_up, _ = best(lambda: gp.set_hyper(h), 1)
    t_gr, (lZ, dlZ) = best(lambda: gp.loglikelihood(True), 1)
    Xs = np.random.RandomState(1).rand(4096, 1)*64
    gp.posterior(Xs[:64])
    t_pr, _ = best(lambda: gp.posterior(Xs), 1)
    say(config='C5-exact', workload='SE+Periodic d=1 N=65536 on ONE GPU: update, loglikelihood(True), posterior(4096)',
        first_add_data_s=t_first, update_s=t_up, grad_s=t_gr, eval_s=t_up + t_gr,
        eff_fp64_tflops=float(n)**3/(t_up + t_gr)/1e12, update_tflops=float(n)**3/3/t_up/1e12,
        predict_points_per_s=len(Xs)/t_pr, lZ=lZ, dlZ_finite=bool(np.all(np.isfinite(dlZ))))


def c5_fitc():
    n, p, d = 1 << 20, 2048, 8
    X, y = problem(n, d)
    U = np.random.RandomState(3).rand(p, d)
    gp = pygp.inference.FITC(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [0.6]*d), 0.0, U)
    t0 = time.perf_counter()
    gp.add_data(X, y)
    t_first = time.perf_counter() - t0
    h = gp.get_hyper()
    gp.loglikelihood(True)
    t_up, _ = best(lambda: gp.set_hyper(h), 2)
    t_gr, (lZ, dlZ) = best(lambda: gp.loglikelihood(True), 2)
    Xs = np.random.RandomState(1).rand(65536, d)
    gp.posterior(Xs[:1024])
    t_pr, _ = best(lambda: gp.posterior(Xs), 2)
    say(config='C5-fitc', workload='FITC SE-ARD d=8, M=2048 pseudo-inputs, N=2^20: update, loglikelihood(True), posterior(65536)',
        first_add_data_s=t_first, update_s=t_up, grad_s=t_gr, eval_s=t_up + t_gr,
        eff_fp64_tflops_8M2N=8.0*p*p*n/(t_up + t_gr)/1e12, predict_points_per_s=len(Xs)/t_pr, lZ=lZ,
        dlZ_finite=bool(np.all(np.isfinite(dlZ))))


def card():
    import subprocess
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    return subprocess.check_output(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader']).decode().strip()


def c5_fitc_pseudo():
    """The C5-fitc shape with d lZ / d U: loglikelihood(True) and loglikelihood(True, pseudoinputs=True)
    alternating, then one profiled call for the contraction kernel's own time (the only PC_GRAM launch
    of a gradient call)."""
    n, p, d = 1 << 20, 2048, 8
    X, y = problem(n, d)
    U = np.random.RandomState(3).rand(p, d)
    gp = pygp.inference.FITC(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [0.6]*d), 0.0, U)
    gp.add_data(X, y)
    gp.loglikelihood(True)
    gp.loglikelihood(True, pseudoinputs=True)
    t_hyp, t_pse = [], []
    for _ in range(4):
        t0 = time.perf_counter()
        gp.loglikelihood(True)
        t_hyp.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        gp.loglikelihood(True, pseudoinputs=True)
        t_pse.append(time.perf_counter() - t0)
    ctx = _lib.context()
    ctx.profile(True)
    gp.loglikelihood(True, pseudoinputs=True)
    launches, kern_ms, _ = ctx.profile_read(1)        # PC_GRAM: pseudo_gram_kernel
    ctx.profile(False)
    # algorithmic bytes: Bt and T2 once (n x p doubles each) plus Cuu, the inputs and alpha, q
    nbytes = 16.0*n*p + 8.0*p*p + 8.0*(n + p)*d + 16.0*n
    # FP64 operations per (pseudo-input, column) entry, counted from the SE instantiation's source: weight 5,
    # distance 3 d, exp 11, gradient 4 d
    flops = (16.0 + 7*d)*p*(n + p)
    hbm_ms, fp64_ms = nbytes/7.7e12*1e3, flops/33.7e12*1e3   # data-sheet HBM3e; measured DFMA (profiles/fp64_peak.json)
    say(config='C5-fitc-pseudo', workload='FITC SE-ARD d=8, M=2048, N=2^20: loglikelihood(True) vs loglikelihood(True, pseudoinputs=True), alternating',
        card=card(), grad_s=sorted(t_hyp), grad_pseudo_s=sorted(t_pse),
        added_ms_median=(float(np.median(t_pse)) - float(np.median(t_hyp)))*1e3,
        pseudo_kernel_launches=launches, pseudo_kernel_ms=kern_ms, algorithmic_gb=nbytes/1e9, fp64_gflop=flops/1e9,
        hbm_bound_ms=hbm_ms, fp64_bound_ms=fp64_ms, bound='fp64' if fp64_ms > hbm_ms else 'hbm',
        share_of_bound=max(hbm_ms, fp64_ms)/kern_ms, target_added_ms=20.0)


def next_rows():
    """The SURVEY 8f rows at a working size: input-gradient predict (N1), joint posterior + draws (N3),
    incremental update (N4), DTC (N4), on N = 8192, d = 8."""
    n, d = 8192, 8
    X, y = problem(n + 64, d)
    Xs = np.random.RandomState(1).rand(4096, d)
    mk = lambda: pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [0.5*np.sqrt(d)]*d), 0.0)
    gp = mk()
    gp.add_data(X[:n], y[:n])
    gp.posterior(Xs[:64], grad=True)
    t_pg, _ = best(lambda: gp.posterior(Xs, grad=True), 2)
    t_p, _ = best(lambda: gp.posterior(Xs), 2)
    gp._full_posterior(Xs[:64])
    t_full, _ = best(lambda: gp._full_posterior(Xs[:1024]), 2)
    t_smp, _ = best(lambda: gp.sample(Xs[:1024], 8, rng=0), 2)
    t_full_upd, _ = best(lambda: gp.set_hyper(gp.get_hyper()), 2)
    t_inc = []
    for i in range(8):                                   # one datum at a time, as a BO loop / SMC does
        t0 = time.perf_counter()
        gp.add_data(X[n + i:n + i + 1], y[n + i:n + i + 1])
        t_inc.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    gp.add_data(X[n + 8:n + 64], y[n + 8:n + 64])        # a block of 56
    t_inc56 = time.perf_counter() - t0
    ref = mk()
    ref.add_data(X, y)
    err = abs(ref.loglikelihood() - gp.loglikelihood())/abs(ref.loglikelihood())
    U = np.random.RandomState(3).rand(512, d)
    dtc = pygp.inference.DTC(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [0.6]*d), 0.0, U)
    Xb, yb = problem(262144, d)
    dtc.add_data(Xb, yb)
    dtc.loglikelihood(True)
    h = dtc.get_hyper()
    t_dtc, _ = best(lambda: (dtc.set_hyper(h), dtc.loglikelihood(True)), 2)
    say(config='next-rows', workload='ExactGP SE-ARD d=8 N=8192: N1 predict with input-gradients, N3 joint posterior / draws, '
        'N4 incremental update; DTC M=512 N=262144',
        predict_points_per_s=len(Xs)/t_p, predict_grad_points_per_s=len(Xs)/t_pg,
        full_posterior_1024_ms=t_full*1e3, sample_8x1024_ms=t_smp*1e3,
        full_update_ms=t_full_upd*1e3, incremental_update_1_ms=float(np.median(t_inc))*1e3,
        incremental_update_56_ms=t_inc56*1e3, incremental_vs_full_lZ_rel_err=err, dtc_eval_ms=t_dtc*1e3)


def main():
    what = sys.argv[1:] or ['c1', 'c2', 'c4', 'c5_fitc', 'c5_exact', 'next_rows']
    _lib.context()
    for w in what:
        globals()[w]()


if __name__ == '__main__':
    main()
