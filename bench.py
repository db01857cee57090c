#!/usr/bin/env python
"""
bench.py -- headline benchmark of the B200 exact-GP hot path.

Metric (BASELINE.json): ExactGP loglike+grad evaluations/s at N=32768, FP64.
Workload = configs[2]: Matern-5/2 ARD, d=16, N=32768 on one GPU; one "step" is
one optimiser objective evaluation = set_hyper (Gram + Cholesky + solve) +
loglikelihood(grad=True).  Synthetic data per SURVEY.md section 8d.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 (torchrun, one rank per GPU): the N = 32768 evaluation fits one GPU and its
optimiser loop is sequential ("replicas only", DESIGN.md section 6) -- `value` is the
aggregate evaluations/s of independent replicas (restarts / chains), weak scaling.
The paths that DO partition are measured beside it at every N (same JSON line):
  dist_chol_n65536   BASELINE configs[4]: SE + Periodic, N = 65536 -- block-column
                     distributed Cholesky + block-column gradient (csrc/dist.cu, NCCL panel
                     broadcast), seconds and speed-up over the one-GPU evaluation
  predict_strong     a FIXED total of test points (default 1 Mi) through
                     sharding.sharded_posterior, host arrays in, all-gather included
  mcmc_4096x2048     BASELINE configs[3]: 4096 hyper samples x N = 2048 through
                     sharding.sharded_batched_loglike (batched Cholesky, sharded by sample)

--impl reference times the reference's algorithm on the host cores (the numpy
oracle port; the reference itself is Python 2 and cannot travel to the GPU box) with
all host threads, at N = 8192 (SURVEY.md 8d), N^3-extrapolated (x64) to the metric's N
and labelled so, plus a bare LAPACK dpotrf + dpotri lower bound.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

if 'reference' in sys.argv:
    # the reference arm is a CPU job: every host core, set before numpy loads its BLAS (torchrun exports
    # OMP_NUM_THREADS=1 to the ranks, which made round 1's N > 1 reference arm silently single-threaded)
    for _k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_k] = str(os.cpu_count() or 1)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'exactgp_loglike_grad_evals_per_s_N32768_fp64'
UNIT = 'evals/s'


def problem(n, d, seed=0):
    rng = np.random.RandomState(seed)
    X = rng.rand(n, d)
    y = np.sin(3*X.sum(1)) + 0.1*rng.randn(n)
    return X, y


def base_hypers(d):
    # [log sn, log sf, log ell_1..d, mean]; ell = 0.5 sqrt(d) (SURVEY.md 8d)
    return np.r_[np.log(0.1), 0.0, np.log(0.5*np.sqrt(d))*np.ones(d), 0.0]


def step_hypers(d, step, rank):
    rng = np.random.RandomState(1000 + 97*rank + step)
    return base_hypers(d) + 0.02*rng.randn(d + 3)


# ---------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


def dist_setup(n_gpus):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    return rank, world, local


def barrier(world):
    import torch
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


# ---------------------------------------------------------------------------
def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is a CPU job on rank 0
    and gets every core (SURVEY.md 8d).  Must run before numpy / scipy load their BLAS."""
    n = str(os.cpu_count() or 1)
    for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[k] = n
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(int(n))
    except Exception:
        pass


def cpu_reference_eval(n_s, d, budget_s, max_steps, rank=0):
    """The reference algorithm (oracle port of exact.py:50-55,118-143) on the host cores:
    set_hyper + loglikelihood(True) at a bounded N.  One warm-up at N/4 (BLAS threads, page
    faults), then timed evaluations at n_s until `max_steps` or the time budget is used.
    Returns (seconds per evaluation, evaluations timed)."""
    from oracle.pygp_oracle import make_kernel, OExactGP
    ell = list(0.5*np.sqrt(d)*np.ones(d))

    def model(n):
        X, y = problem(n, d)
        gp = OExactGP(0.1, make_kernel(('matern', 1.0, ell, 5)), 0.0)
        gp.add_data(X, y)
        return gp
    w = model(max(256, n_s//4))
    w.set_hyper(step_hypers(d, 0, rank))
    w.loglikelihood(True)
    del w
    gp = model(n_s)
    times, t_start = [], time.perf_counter()
    for s in range(max(1, max_steps)):
        h = step_hypers(d, 1 + s, rank)
        t0 = time.perf_counter()
        gp.set_hyper(h)
        gp.loglikelihood(True)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start + times[-1] > budget_s:
            break
    return float(np.mean(times)), len(times)


def lapack_lower_bound(n_l, n):
    """Bare LAPACK dpotrf + dpotri (what any CPU implementation of loglike+grad must at least do:
    the factor and the explicit inverse, N^3 flops) on an SPD matrix of order n_l, N^3-scaled to n.
    n_l = n (16 GiB at 32768, ~minutes of CPU) under --cpu-full, else a bounded n_l."""
    from scipy.linalg import lapack
    rng = np.random.RandomState(0)
    A = rng.rand(n_l, 64)
    K = A @ A.T
    K[np.diag_indices(n_l)] += n_l
    K = np.asfortranarray(K)
    t0 = time.perf_counter()
    c, info = lapack.dpotrf(K, lower=1, overwrite_a=1)
    t1 = time.perf_counter()
    inv, info2 = lapack.dpotri(c, lower=1, overwrite_c=1)
    t2 = time.perf_counter()
    assert info == 0 and info2 == 0
    scale = (float(n)/n_l)**3
    return {'n': n_l, 'dpotrf_s': t1 - t0, 'dpotri_s': t2 - t1, 'gflops': n_l**3/(t2 - t0)/1e9,
            'scaled_to_n': n, 'scale': scale, 'seconds_at_n': (t2 - t0)*scale, 'evals_per_s_at_n': 1.0/((t2 - t0)*scale),
            'what': 'scipy.linalg.lapack dpotrf + dpotri, N^3 flops, N^3-scaled x%.0f' % scale}


def host_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get('num_threads', 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline_record(args, budget_s, max_steps):
    n, d, n_s = args.n, args.d, args.cpu_n
    sec, k = cpu_reference_eval(n_s, d, budget_s, max_steps)
    scale = (float(n)/n_s)**3
    sec_n = sec*scale
    lap = lapack_lower_bound(n if args.cpu_full else min(n, args.lapack_n), n)
    sample = ('oracle numpy port of exact.py:50-55,118-143 (set_hyper + loglikelihood(True)), Matern-5/2 ARD d=%d: '
              '%.2f s/eval at N=%d (%d timed), N^3-EXTRAPOLATED x%.0f to N=%d = %.0f s (the reference itself needs '
              '>72 GiB at N=32768; its O(N^2) per-hyper loop makes N^3 scaling pessimistic for the CPU by <2x); '
              'bare LAPACK lower bound: %.0f s' % (d, sec, n_s, k, scale, n, sec_n, lap['seconds_at_n']))
    return {'value': 1.0/sec_n, 'unit': UNIT, 'cores': host_threads(), 'kind': 'port', 'sample': sample,
            'sample_n': n_s, 'sample_s_per_eval': sec, 'sample_evals': k, 'extrapolation_factor': scale,
            'lapack_lower_bound': lap}, sec_n, k


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    use_all_host_threads()
    cpu, sec_n, k = cpu_baseline_record(args, args.cpu_budget, args.steps)
    value = cpu['value']
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': k, 'warmup': 1, 'steps_requested': args.steps, 'ms_per_step': sec_n*1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'ExactGP Matern-5/2 ARD d=%d N=%d loglike+grad (CPU sample N=%d, N^3-extrapolated x%.0f; '
                               'timed evaluations bounded by a %.0f s budget)'
                               % (args.d, args.n, args.cpu_n, cpu['extrapolation_factor'], args.cpu_budget)},
        'cpu_baseline': cpu,
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
def run_ours(args):
    import torch
    rank, world, local = dist_setup(args.gpus)
    os.environ['PYGP_B200_DEVICE'] = str(local)
    torch.cuda.set_device(local)
    import pygp_b200 as pygp
    from pygp_b200 import _lib
    ctx = _lib.context(local)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device('cuda', local))
    n, d, K, W = args.n, args.d, args.steps, args.warmup
    nh = d + 3

    # FP64 roofline denominator: cuBLAS DGEMM measured in this run (the driver's
    # MEASURED_PEAKS.json carries HBM and bf16 only)
    def dgemm_peak():
        m = 8192
        a = torch.randn(m, m, dtype=torch.float64, device='cuda')
        b = torch.randn(m, m, dtype=torch.float64, device='cuda')
        c = torch.empty(m, m, dtype=torch.float64, device='cuda')
        best = 1e30
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b, c
        torch.cuda.empty_cache()
        return 2*m**3/(best*1e-3)/1e12
    fp64_peak = dgemm_peak()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    hbm_src = 'MEASURED_PEAKS.json' if 'hbm_gbs' in peaks else 'fallback B200_PROFILING.md'

    # pinned host inputs (e2e copies them every step)
    X, y = problem(n, d)
    Xp = torch.empty((n, d), dtype=torch.float64).pin_memory()
    yp = torch.empty((n,), dtype=torch.float64).pin_memory()
    Xp.numpy()[:] = X
    yp.numpy()[:] = y
    Xh, yh = Xp.numpy(), yp.numpy()

    def make_gp():
        ell = list(0.5*np.sqrt(d)*np.ones(d))
        return pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1), pygp.kernels.Matern(1.0, ell, 5), 0.0)

    # ---- value: inputs resident in HBM ------------------------------------------------
    gp = make_gp()
    gp.add_data(Xh, yh)
    for s in range(W):
        gp.set_hyper(step_hypers(d, s, rank))
        gp.loglikelihood(True)
    ctx.profile(True)
    barrier(world)
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record(stream)
        t0 = time.perf_counter()
        for s in range(K):
            gp.set_hyper(step_hypers(d, W + s, rank))
            lZ, dlZ = gp.loglikelihood(True)
        e1.record(stream)
        ctx.sync()
        wall = time.perf_counter() - t0
    dev_s = e0.elapsed_time(e1)*1e-3
    launches = ctx.launch_count - l0
    names = ['gemm', 'gram', 'trace', 'potrf_base', 'trsm_base', 'other']
    prof = {nm: ctx.profile_read(i) for i, nm in enumerate(names)}
    ctx.profile(False)
    barrier(world)
    t_max = max_over_ranks(max(dev_s, 0.0), world)
    value = world*K/t_max
    assert np.isfinite(lZ) and np.all(np.isfinite(dlZ))
    if args.dump_outputs and rank == 0:
        # what the last timed step returned to its caller, for output-by-output comparison of two builds
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'lZ.npy'), np.asarray(lZ, dtype=np.float64))
        np.save(os.path.join(args.dump_outputs, 'dlZ.npy'), np.asarray(dlZ, dtype=np.float64))

    # ---- e2e: public API with host buffers, H2D of X, y and D2H of (lZ, dlZ) each step --
    del gp
    for s in range(min(W, 1)):
        g2 = make_gp()
        g2.add_data(Xh, yh)
        g2.loglikelihood(True)
        del g2
    barrier(world)
    t0 = time.perf_counter()
    for s in range(K):
        g2 = make_gp()
        g2.set_hyper(step_hypers(d, W + s, rank))
        g2.add_data(Xh, yh)
        lZ2, dlZ2 = g2.loglikelihood(True)
        del g2
    ctx.sync()
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    e2e = {'value': world*K/e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': int(8*(n*d + n + nh)),
           'd2h_bytes_per_step': int(8*(1 + nh)), 'timed': 'wall clock around ExactGP() + add_data + '
           'loglikelihood(True), device allocation included'}

    # ---- secondary: sharded predict and Gram build ------------------------------------
    gp = make_gp()
    gp.add_data(Xh, yh)
    extra = {}
    m_loc = args.predict_pts            # per rank: test points shard with no collective (weak scaling, like `value`)
    Xs = torch.rand(m_loc, d, dtype=torch.float64, device='cuda',
                    generator=torch.Generator('cuda').manual_seed(1 + rank))
    mu = torch.empty(m_loc, dtype=torch.float64, device='cuda')
    s2 = torch.empty(m_loc, dtype=torch.float64, device='cuda')
    L = _lib.lib()

    def predict():
        _lib.check(ctx, L.pgp_exact_predict_dev(gp._dev.handle, Xs.data_ptr(), m_loc, mu.data_ptr(), s2.data_ptr()))
    predict()
    barrier(world)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record(stream)
    predict()
    pe1.record(stream)
    ctx.sync()
    p_s = max_over_ranks(pe0.elapsed_time(pe1)*1e-3, world)
    extra['predict_points_per_s'] = m_loc*world/p_s
    extra['predict_fp64_tflops_per_gpu'] = m_loc*float(n)*n/p_s/1e12
    extra['predict_points'] = m_loc*world
    Xs_pin = torch.empty((m_loc, d), dtype=torch.float64).pin_memory()      # pinned host test points
    Xs_pin.copy_(Xs)
    Xs_h = Xs_pin.numpy()
    barrier(world)
    t0 = time.perf_counter()
    gp.posterior(Xs_h)
    extra['predict_points_per_s_e2e'] = m_loc*world/max_over_ranks(time.perf_counter() - t0, world)
    del Xs, mu, s2

    # ---- the paths that partition (SURVEY 8e), measured at every N ------------------------
    if not args.no_scale_legs:
        from pygp_b200 import sharding, distchol
        try:
            # (1) predict, STRONG scaling: a fixed total of test points through sharding.sharded_posterior
            #     (host array in, per-rank slice H2D + predict + D2H, all-gather of (mu, s2) included)
            m_tot = args.predict_total
            Xt = np.random.RandomState(7).rand(m_tot, d)
            sharding.sharded_posterior(gp, Xt[:world*256])                 # warm-up (buffers, NCCL channel)
            barrier(world)
            t0 = time.perf_counter()
            mu_t, s2_t = sharding.sharded_posterior(gp, Xt)
            t_pred = max_over_ranks(time.perf_counter() - t0, world)
            assert mu_t.shape == (m_tot,) and np.all(np.isfinite(mu_t)) and np.all(s2_t > 0)
            extra['predict_strong'] = {
                'points_total': m_tot, 'seconds': t_pred, 'points_per_s': m_tot/t_pred,
                'fp64_tflops_per_gpu': m_tot/world*float(n)*n/t_pred/1e12,
                'what': 'sharding.sharded_posterior: N=%d d=%d model replicated, %d test points split over %d rank(s), '
                        'host arrays, all-gather of (mu, s2) included' % (n, d, m_tot, world)}
            del Xt, mu_t, s2_t
        except Exception as e:                 # a failed leg must not cost the headline line
            extra['predict_strong'] = {'error': '%s: %s' % (type(e).__name__, e)}
    kern_main = gp._kernel
    del gp

    if rank == 0:
        ng = min(n, 32768)
        out = torch.empty(ng, ng, dtype=torch.float64, device='cuda')

        def gram_rate(kern, Xg):
            Xd = torch.tensor(Xg, device='cuda')
            hyp = _lib.as_f64(kern.get_hyper())
            spec = kern._spec()

            def gram():
                _lib.check(ctx, L.pgp_gram_dev(ctx.handle, spec, _lib.ptr(hyp), Xd.data_ptr(), ng, None, ng,
                                               out.data_ptr()))
            gram()
            ctx.profile(True)
            gram()
            cnt, ms, work = ctx.profile_read(1)
            ctx.profile(False)
            return work/ms/1e6, ms, work
        # the workload's kernel (FP64-pipe bound: ~(2d + 45) DP instructions per entry, DESIGN.md 4) ...
        gbs, ms, work = gram_rate(kern_main, X[:ng])
        extra['gram_build_GBps'] = gbs
        extra['gram_build_hbm_frac'] = gbs/hbm_peak
        extra['gram_build'] = 'Kernel.get(X) full square N=%d d=%d: %.1f MB written in %.3f ms' % (ng, d, work/1e6, ms)
        # ... and the d=1 SE kernel of configs C1 / C5, where the 8 B / entry written is the bound
        gbs1, ms1, work1 = gram_rate(pygp.kernels.SE(1.0, 0.1, ndim=1), X[:ng, :1])
        extra['gram_build_d1_GBps'] = gbs1
        extra['gram_build_d1_hbm_frac'] = gbs1/hbm_peak
        extra['gram_build_d1'] = 'SE iso d=1 N=%d: %.1f MB written in %.3f ms' % (ng, work1/1e6, ms1)
        del out

    if not args.no_scale_legs:
        from pygp_b200 import sharding, distchol
        ctx.sync()
        try:
            # (2) batched MCMC (BASELINE configs[3]): 4096 hyper samples x N = 2048 SE-ARD d = 8 through
            #     sharding.sharded_batched_loglike: B / G samples per rank, results all-gathered
            nb_, db_, B_ = 2048, 8, 4096
            Xb, yb = problem(nb_, db_, seed=2)
            gb = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1),
                                        pygp.kernels.SE(1.0, list(0.5*np.sqrt(db_)*np.ones(db_))), 0.0)
            gb.add_data(Xb, yb)
            H = gb.get_hyper() + np.random.RandomState(2).uniform(-0.5, 0.5, size=(B_, gb.nhyper))
            sharding.sharded_batched_loglike(gb, H[:world*8])              # warm-up
            barrier(world)
            t0 = time.perf_counter()
            lz_b = sharding.sharded_batched_loglike(gb, H)
            t_b = max_over_ranks(time.perf_counter() - t0, world)
            assert lz_b.shape == (B_,) and np.all(np.isfinite(lz_b))
            extra['mcmc_4096x2048'] = {
                'samples': B_, 'n': nb_, 'seconds': t_b, 'samples_per_s': B_/t_b,
                'potrf_tflops_per_gpu': B_/world*float(nb_)**3/3/t_b/1e12,
                'what': 'sharding.sharded_batched_loglike: %d hyper vectors x N=%d SE-ARD d=%d, sharded by sample over '
                        '%d rank(s) (batched Gram + Cholesky + solve), all-gather of lZ included' % (B_, nb_, db_, world)}
            del gb, lz_b
        except Exception as e:
            extra['mcmc_4096x2048'] = {'error': '%s: %s' % (type(e).__name__, e)}

        try:
            torch.cuda.empty_cache()
            # (3) C5 (BASELINE configs[4]): SE + Periodic, N = 65536.  One-GPU evaluation (every rank runs it on its
            #     own GPU) and the block-column distributed evaluation over all ranks (csrc/dist.cu)
            n5, nb5 = args.c5_n, args.c5_nb
            rng5 = np.random.RandomState(0)
            X5 = np.sort(rng5.rand(n5, 1), axis=0)*64
            y5 = np.sin(3*X5.sum(1)) + 0.1*rng5.randn(n5)
            mk5 = lambda: pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1),
                                                 pygp.kernels.SE(1.0, 0.5, 1) + pygp.kernels.Periodic(0.5, 1.0, 0.25), 0.0)
            g5 = mk5()
            g5.add_data(X5, y5)                                            # upload + first factorisation (untimed)
            h5 = g5.get_hyper()
            ctx.sync()
            t0 = time.perf_counter()
            g5.set_hyper(h5 + 0.01)
            ctx.sync()
            t_u1 = time.perf_counter() - t0
            t0 = time.perf_counter()
            lZ5, dlZ5 = g5.loglikelihood(True)
            t_g1 = time.perf_counter() - t0
            t_u1, t_g1 = max_over_ranks(t_u1, world), max_over_ranks(t_g1, world)
            c5 = {'n': n5, 'nb': nb5, 'update_1gpu_s': t_u1, 'loglike_grad_1gpu_s': t_g1,
                  'eval_1gpu_s': t_u1 + t_g1, 'eval_1gpu_tflops': float(n5)**3/(t_u1 + t_g1)/1e12}
            del g5                                                         # its 2 N^2 gradient buffers return to the pool
            g5 = mk5()
            g5.add_data(X5, y5)
            g5._likelihood.set_hyper((h5 + 0.01)[:1]); g5._kernel.set_hyper((h5 + 0.01)[1:-1]); g5._mean = float(h5[-1] + 0.01)
            for rep in range(2):                                           # first pass: buffers, NCCL channels
                barrier(world)
                t0 = time.perf_counter()
                distchol.distributed_update(g5, nb=nb5)
                ctx.sync()
                t_ud = max_over_ranks(time.perf_counter() - t0, world)
                t0 = time.perf_counter()
                lZd, dlZd = distchol.distributed_loglikelihood(g5, True, nb=nb5)
                t_gd = max_over_ranks(time.perf_counter() - t0, world)
            c5.update({'update_s': t_ud, 'loglike_grad_s': t_gd, 'eval_s': t_ud + t_gd,
                       'speedup_vs_1gpu': (t_u1 + t_g1)/(t_ud + t_gd), 'update_speedup_vs_1gpu': t_u1/t_ud,
                       'loglike_grad_speedup_vs_1gpu': t_g1/t_gd,
                       'aggregate_tflops': float(n5)**3/(t_ud + t_gd)/1e12,
                       'lZ_rel_diff_vs_1gpu': abs(lZd - lZ5)/abs(lZ5),
                       'dlZ_rel_diff_vs_1gpu': float(np.abs(dlZd - dlZ5).max()/np.abs(dlZ5).max()),
                       'what': 'SE + Periodic d=1, N=%d: ExactGP._update + loglikelihood(True); 1 GPU = pgp_exact_update / '
                               '_loglike, %d rank(s) = pgp_dist_exact_update / _loglike (block columns of %d, NCCL panel '
                               'broadcast, block-column gradient + one all-reduce)' % (n5, world, nb5)})
            # parity of the distributed evaluation with the one-GPU one, at the north-star tolerances: reported, not
            # asserted (a benchmark line with `parity_ok: false` is worth more than no line; tests/test_multigpu.py asserts it)
            c5['parity_ok'] = bool(c5['lZ_rel_diff_vs_1gpu'] <= 1e-10 and c5['dlZ_rel_diff_vs_1gpu'] <= 1e-8)
            extra['dist_chol_n65536'] = c5
            del g5
        except Exception as e:
            extra['dist_chol_n65536'] = {'error': '%s: %s' % (type(e).__name__, e)}

    # ---- CPU baseline (rank 0, N = 1 only): ONE evaluation of the oracle port at N = 8192 -----------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        use_all_host_threads()
        cpu, _, _ = cpu_baseline_record(args, 0.0, 1)

    if rank == 0:
        g_l, g_ms, g_work = prof['gemm']
        achieved = g_work/(g_ms*1e-3)/1e12 if g_ms > 0 else 0.0
        # roofline.traffic: DRAM bytes of ONE launch of the dominant kernel from the committed ncu --set full
        # capture (an 8192^3 launch; the launches of a step have many shapes, so the capture's own algorithmic
        # bytes are given beside it in traffic_detail)
        fp64_file = None
        try:
            fp64_file = json.load(open(os.path.join(ROOT, 'profiles', 'fp64_peak.json')))
        except Exception:
            pass
        traffic, traffic_detail = None, None
        try:
            traffic_detail = json.load(open(os.path.join(ROOT, 'profiles', 'gemm_traffic.json')))
            traffic = traffic_detail['dram_bytes_per_launch']
        except Exception:
            pass
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': t_max/K*1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': 'ExactGP Matern-5/2 ARD d=%d N=%d: set_hyper (Gram+Cholesky+solve) + '
                                   'loglikelihood(grad=True) [BASELINE configs[2]]' % (d, n),
                       'l2': 'working set %.1f GiB per evaluation >> 126 MB L2 (no flush needed)' % (3*n*n*8/2**30),
                       'parallelism': 'replicas x%d (independent hyper vectors per GPU)' % world},
            'eff_fp64_tflops_per_gpu': float(n)**3*K/dev_s/1e12,
            'eff_fp64_frac_of_dgemm': float(n)**3*K/dev_s/1e12/fp64_peak,
            'wall_s': wall, 'device_s': dev_s,
            'roofline': {'bound': 'tensor', 'kernel': 'gemm_nt_kernel (FP64 DMMA)', 'achieved': achieved,
                         'peak': fp64_peak, 'unit': 'TFLOP/s', 'frac': achieved/fp64_peak if fp64_peak else None,
                         'traffic': traffic, 'traffic_detail': traffic_detail, 'launches': g_l, 'avg_launch_ms': g_ms/max(g_l, 1),
                         'share_of_step': g_ms*1e-3/dev_s,
                         'peak_source': 'cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 '
                                        'entry; nominal 37 TFLOP/s); HBM %s' % hbm_src,
                         'fp64_peaks_on_file': fp64_file,
                         'frac_of_dmma_issue_peak': (achieved/fp64_file['dmma_tflops']
                                                     if fp64_file and fp64_file.get('dmma_tflops') else None)},
            'kernel_ms_per_step': {nm: prof[nm][1]/K for nm in names},
            'kernel_launches_per_step': {nm: prof[nm][0]/K for nm in names},
            'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': int(launches),
            'clocks': clocks.summary(), 'lZ_last': float(lZ),
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--n', type=int, default=32768)
    ap.add_argument('--d', type=int, default=16)
    ap.add_argument('--cpu-n', type=int, default=8192, dest='cpu_n', help='N of the CPU sample (SURVEY 8d: 8192)')
    ap.add_argument('--cpu-budget', type=float, default=150.0, dest='cpu_budget',
                    help='reference arm: stop timing further evaluations after this many seconds')
    ap.add_argument('--lapack-n', type=int, default=16384, dest='lapack_n',
                    help='order of the dpotrf+dpotri lower-bound sample (N^3-scaled to --n)')
    ap.add_argument('--cpu-full', action='store_true', dest='cpu_full', help='LAPACK lower bound at the full N')
    ap.add_argument('--predict-total', type=int, default=1 << 20, dest='predict_total',
                    help='test points of the strong-scaling predict leg (total over all ranks)')
    ap.add_argument('--c5-n', type=int, default=65536, dest='c5_n')
    ap.add_argument('--c5-nb', type=int, default=512, dest='c5_nb')
    ap.add_argument('--no-scale-legs', action='store_true', dest='no_scale_legs',
                    help='skip dist_chol_n65536 / predict_strong / mcmc_4096x2048')
    ap.add_argument('--predict-pts', type=int, default=16384, dest='predict_pts', help='test points per rank')
    ap.add_argument('--no-cpu', action='store_true', dest='no_cpu')
    ap.add_argument('--dump-outputs', dest='dump_outputs', metavar='DIR',
                    help='write lZ and dlZ of the last timed step (rank 0) as DIR/lZ.npy, DIR/dlZ.npy in float64')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
