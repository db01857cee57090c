"""Incremental FITC / DTC add_data on the GPU (pgp_fitc_append_inc) against the
full update at SE-ARD d = 8, M = 2048 pseudo-inputs, N = 2^20 rows: the append
time for m = 1, 8, 64 new rows (host clock around calls that end in a stream
synchronise), the rank-update kernels' device time from CUDA events, end-to-end
FITC.add_data of one row with the host's concatenation timed on its own, and
the full pgp_fitc_update.  Writes profiles/r07_fitc_inc.txt (or the path given
as the first argument).

    python tools/fitc_inc_probe.py [out.txt]
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

PC_POTRF, PC_TRSM = 3, 4   # profile classes of the rank-m update's panel chain and of its row application
D, M, N = 8, 2048, 1 << 20
LINES = []


def out(s):
    print(s, flush=True)
    LINES.append(s)


def card():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    return subprocess.check_output(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader']).decode().strip()


def rows(rng, m):
    X = rng.rand(m, D)
    return X, np.sin(3*X.sum(1)) + 0.1*rng.randn(m)


def timed(fn):
    _lib.context().sync()
    t0 = time.perf_counter()
    fn()
    _lib.context().sync()
    return time.perf_counter() - t0


def stats(ts):
    ts = np.asarray(ts)*1e3
    return 'median %.3f ms  min %.3f  max %.3f  (%d runs)' % (np.median(ts), ts.min(), ts.max(), len(ts))


def probe(dtc):
    name = 'DTC' if dtc else 'FITC'
    rng = np.random.RandomState(0)
    X, y = rows(rng, N)
    U = rng.rand(M, D)
    cls = pygp.inference.DTC if dtc else pygp.inference.FITC
    # DTC's Kuu + Kux Kxu / sn2 + su2 I (su2 = 1e-6 sn2) is not positive definite in FP64 at this N with the
    # smooth FITC kernel; shorter length-scales keep it so
    ell = 0.5 if dtc else 0.5*np.sqrt(D)
    gp = cls(pygp.likelihoods.Gaussian(0.1), pygp.kernels.SE(1.0, [ell]*D), 0.0, U)
    t = timed(lambda: gp.add_data(X, y))
    out('%s  SE-ARD d=%d (length-scales %.3g)  M=%d  N=%d' % (name, D, ell, M, N))
    out('  create + full update (first call)          %.3f s' % t)
    lib, h = _lib.lib(), gp._dev.handle
    hyp = _lib.as_f64(gp.get_hyper())
    ctx = gp._dev.ctx
    ts = [timed(lambda: _lib.check(ctx, lib.pgp_fitc_update(h, _lib.ptr(hyp)))) for _ in range(3)]
    out('  pgp_fitc_update (full, N rows)             ' + stats(ts))

    # end-to-end GP.add_data of one row (the first append reallocates the row buffers with slack)
    Xa, ya = rows(rng, 1)
    out('  first add_data(1 row), with reallocation   %.3f ms' % (1e3*timed(lambda: gp.add_data(Xa, ya))))
    h0 = gp._dev
    ts = []
    for _ in range(20):
        Xa, ya = rows(rng, 1)
        ts.append(timed(lambda: gp.add_data(Xa, ya)))
    assert gp._dev is h0, 'add_data left the incremental path'
    out('  FITC.add_data(1 row) end to end            ' + stats(ts))
    Xh, yh = gp.data
    ts = []
    for _ in range(20):
        t0 = time.perf_counter()
        _ = np.r_[Xh, Xa], np.r_[yh, ya]
        ts.append(time.perf_counter() - t0)
    out('    of which the host np.r_ of X, y          ' + stats(ts))
    lz_inc = gp.loglikelihood()

    # the library call alone, m = 1, 8, 64 (the host data is not kept in step from here on)
    for m in (1, 8, 64):
        ts = []
        for _ in range(20 if m < 64 else 10):
            Xm, ym = rows(rng, m)
            Xm, ym = _lib.as_f64(Xm, 2), _lib.as_f64(ym)
            ts.append(timed(lambda: _lib.check(ctx, lib.pgp_fitc_append_inc(h, _lib.ptr(Xm), _lib.ptr(ym), m))))
        out('  pgp_fitc_append_inc m=%-2d                   %s' % (m, stats(ts)))
    for m in (1, 8, 64):
        ctx.profile(True)
        Xm, ym = rows(rng, m)
        Xm, ym = _lib.as_f64(Xm, 2), _lib.as_f64(ym)
        _lib.check(ctx, lib.pgp_fitc_append_inc(h, _lib.ptr(Xm), _lib.ptr(ym), m))
        ctx.sync()
        tot = sum(ctx.profile_read(c)[1] for c in range(6))
        ctx.profile(False)
        out('  m=%-2d all kernels of the append (events)   %.3f ms' % (m, tot))
    out('  lZ after the timed add_data calls: %.12g' % lz_inc)
    del gp, h0
    gc.collect()


def rank_update():
    """pgp_dev_chol_update alone on a p = 2048 factor with one riding row, split into the panel chain
    (one CTA per panel) and the application to the rows below each panel, from CUDA events."""
    import torch
    ctx, lib = _lib.context(), _lib.lib()
    p, ld = M, M
    rng = np.random.RandomState(1)
    B = rng.randn(p, p)
    Lf = np.linalg.cholesky(B.dot(B.T)/p + np.eye(p))
    F0 = np.zeros((p + 1, ld))
    F0[:p, :p] = Lf
    F0[p, :p] = rng.randn(p)
    dF0 = torch.tensor(F0, device='cuda')
    dF = dF0.clone()
    out('rank-m update kernels alone (pgp_dev_chol_update), p = %d, one riding row, %d panels' % (p, p // 64))
    for m in (1, 8, 64):
        ldw = (p + 1 + 15)//16*16
        W0 = torch.tensor(rng.randn(m, ldw)*0.1, device='cuda')
        dW = W0.clone()
        for rep in range(6):                  # rep 0 warms up; the factor is reset before every call
            dF.copy_(dF0)
            dW.copy_(W0)
            torch.cuda.synchronize()
            if rep == 1:
                ctx.profile(True)
            _lib.check(ctx, lib.pgp_dev_chol_update(ctx.handle, dF.data_ptr(), p, ld, 1, dW.data_ptr(), ldw, m))
        ctx.sync()
        (lp, msp, _), (la, msa, _) = ctx.profile_read(PC_POTRF), ctx.profile_read(PC_TRSM)
        ctx.profile(False)
        calls = 5
        out('  m=%-2d per call: panel chain %.3f ms (%d launches, %.2f us per panel), row application %.3f ms '
            '(%d launches, %.2f us per panel)'
            % (m, msp/calls, lp//calls, 1e3*msp/lp, msa/calls, la//calls, 1e3*msa/max(la, 1)))


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles', 'r07_fitc_inc.txt')
    out('# tools/fitc_inc_probe.py -- incremental FITC / DTC add_data vs the full update')
    out('# card (name, power limit, SM clock, max SM clock): ' + card())
    try:
        rank_update()
        for dtc in (False, True):
            probe(dtc)
    finally:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, 'w') as f:
            f.write('\n'.join(LINES) + '\n')


if __name__ == '__main__':
    main()
