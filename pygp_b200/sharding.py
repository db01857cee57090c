"""
Multi-GPU sharding of the parts of the path that partition naturally
(SURVEY.md section 8e): one process per GPU, `torch.distributed` for the
plumbing.

  * predict          -- independent test points: each rank evaluates a contiguous
                        slice on its own replica of the model; the (mu, s2) slices
                        are all-gathered.  No data-path collective.
  * batched hypers   -- independent hyper-parameter samples (learning/sampling.py:146,
                        meta/mcmc.py:75-93): each rank evaluates B/G of them; results
                        all-gathered.  No data-path collective.
  * mixture moments  -- MCMC.posterior (mcmc.py:84-93) over sharded samples needs two
                        small all-reduces: sum mu_i, then sum (s2_i + (mu_i - mu)^2); with
                        input-gradients the same two carry sum dmu_i and
                        sum (ds2_i + 2 (mu_i - mu)(dmu_i - dmu)) along.

The optimiser / slice-sampler loops are sequential: replicas only (one restart or
chain per GPU), nothing to do here.

Every function works without an initialised process group (world size 1) and
with any backend: tensors are staged on the device the backend needs (CUDA for
NCCL, host for gloo -- which is how tests/test_sharding.py runs on CPU).
"""

import numpy as np

__all__ = ['shard_range', 'world', 'all_gather_rows', 'all_reduce_sum', 'sharded_posterior', '_raise_together',
           'sharded_batched_loglike', 'sharded_mixture_posterior']


def world(group=None):
    """(rank, world_size) of the default / given process group; (0, 1) without one."""
    try:
        import torch.distributed as dist
    except ImportError:      # pragma: no cover
        return 0, 1
    if not (dist.is_available() and dist.is_initialized()):
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def shard_range(total, rank, size):
    """Contiguous slice [lo, hi) of `total` items owned by `rank`: the first
    total % size ranks get one extra item (sizes differ by at most one)."""
    base, rem = divmod(int(total), int(size))
    lo = rank*base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _device_for(group):
    import torch
    import torch.distributed as dist
    backend = dist.get_backend(group)
    if 'nccl' not in str(backend):
        return torch.device('cpu')
    # the device the library context computes on (LOCAL_RANK / PYGP_B200_DEVICE), not torch's current
    # device: collectives and compute must share one GPU even if the caller never called set_device
    from . import _lib
    return torch.device('cuda', _lib.context().device)


def all_gather_rows(local, total, group=None):
    """Concatenate per-rank row blocks (rank r holds rows shard_range(total, r, G))
    of a float64 array along axis 0."""
    rank, size = world(group)
    local = np.ascontiguousarray(local, dtype=np.float64)
    if size == 1:
        return local
    import torch
    import torch.distributed as dist
    dev = _device_for(group)
    tail = local.shape[1:]
    counts = [shard_range(total, r, size) for r in range(size)]
    width = max(hi - lo for lo, hi in counts)           # blocks differ by at most one row: pad to equal size
    mine = torch.zeros((width,) + tail, dtype=torch.float64)
    mine[:len(local)] = torch.from_numpy(local)
    mine = mine.to(dev)
    out = torch.empty((size*width,) + tail, dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(out, mine, group=group)
    out = out.cpu().numpy().reshape((size, width) + tail)
    return np.concatenate([out[r, :hi - lo] for r, (lo, hi) in enumerate(counts)], 0)


def all_reduce_sum(x, group=None):
    rank, size = world(group)
    x = np.ascontiguousarray(x, dtype=np.float64)
    if size == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(x.copy()).to(_device_for(group))
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.cpu().numpy()


def _raise_together(err, group=None):
    """Make a rank-local failure global: all-reduce an error flag (MAX) and raise the
    same exception class on every rank, so that nobody is left waiting in the next
    collective.  `err` is None or the exception caught on this rank."""
    rank, size = world(group)
    code = 0 if err is None else (1 if isinstance(err, np.linalg.LinAlgError) else 2)
    if size > 1:
        import torch
        import torch.distributed as dist
        t = torch.tensor([float(code)], dtype=torch.float64, device=_device_for(group))
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        code = int(t.item())
    if code == 0:
        return
    if err is not None:
        raise err
    if code == 1:
        raise np.linalg.LinAlgError('another rank: kernel matrix not positive definite')
    raise RuntimeError('another rank failed in a sharded evaluation')


def sharded_posterior(gp, X, group=None):
    """`gp.posterior(X)` (exact.py:81-97 / fitc.py:122-142) with the rows of X
    split across the ranks; every rank holds an identical model (same data,
    same hypers) and returns the full (mu, s2)."""
    rank, size = world(group)
    X = np.array(X, ndmin=2, dtype=float)
    lo, hi = shard_range(len(X), rank, size)
    err, mu, s2 = None, np.empty(0), np.empty(0)
    try:
        if hi > lo:
            mu, s2 = gp.posterior(X[lo:hi])
    except Exception as e:                # noqa: BLE001 -- re-raised on every rank below
        err = e
    _raise_together(err, group)
    out = all_gather_rows(np.stack([mu, s2], 1), len(X), group)
    return out[:, 0].copy(), out[:, 1].copy()


def _batched(fn_name, gp, hypers, extra):
    """Run pgp_batched_* for the rows `hypers` on this rank's device."""
    import ctypes as C
    from . import _lib
    ctx, L = _lib.context(), _lib.lib()
    Xd, yd = _lib.as_f64(gp._X, 2), _lib.as_f64(gp._y, 1)
    H = _lib.as_f64(hypers, 2)
    B = len(H)
    info = np.zeros(B, dtype=np.int32)
    ip = info.ctypes.data_as(C.POINTER(C.c_int32))
    spec = gp._kernel._spec()
    if fn_name in ('loglike', 'loglike_grad'):
        lZ = np.empty(B)
        dlZ = np.empty((B, H.shape[1])) if fn_name == 'loglike_grad' else None
        _lib.check(ctx, L.pgp_batched_loglike(ctx.handle, spec, _lib.ptr(Xd), _lib.ptr(yd), len(Xd),
                                              _lib.ptr(H), B, _lib.ptr(lZ), None if dlZ is None else _lib.ptr(dlZ), ip))
        lZ[info != 0] = -np.inf       # not positive definite: zero likelihood
        if dlZ is None:
            return lZ
        dlZ[info != 0] = 0.0
        return np.c_[lZ, dlZ]
    Xs = _lib.as_f64(extra, 2)
    mu, s2 = np.empty((B, len(Xs))), np.empty((B, len(Xs)))
    _lib.check(ctx, L.pgp_batched_predict(ctx.handle, spec, _lib.ptr(Xd), _lib.ptr(yd), len(Xd),
                                          _lib.ptr(H), B, _lib.ptr(Xs), len(Xs), _lib.ptr(mu), _lib.ptr(s2), ip))
    if np.any(info):
        raise np.linalg.LinAlgError('sampled hyper-parameters give a non positive definite kernel matrix')
    return mu, s2


def sharded_batched_loglike(gp, hypers, group=None, local_fn=None, grad=False):
    """log marginal likelihood of `gp`'s data under each row of `hypers`
    ((B, nhyper), full GP vectors), the B problems split across the ranks.
    grad=True: returns (lZ (B,), dlZ (B, nhyper)) -- the objective of a multi-restart
    `optimize` (learning/optimization.py:54-62) or of SMC particles in one device call per rank.
    `local_fn(hypers_slice) -> (b,)` [(b, 1 + nhyper) with grad] replaces the device call
    (host-logic tests)."""
    rank, size = world(group)
    hypers = np.array(hypers, ndmin=2, dtype=float)
    lo, hi = shard_range(len(hypers), rank, size)
    fn = local_fn or (lambda h: _batched('loglike_grad' if grad else 'loglike', gp, h, None))
    err, mine = None, (np.empty((0, 1 + hypers.shape[1])) if grad else np.empty(0))
    try:
        if hi > lo:
            mine = fn(hypers[lo:hi])
    except Exception as e:                # noqa: BLE001
        err = e
    _raise_together(err, group)
    out = all_gather_rows(np.asarray(mine, dtype=float), len(hypers), group)
    return (out[:, 0].copy(), out[:, 1:].copy()) if grad else out


def sharded_mixture_posterior(gp, hypers, X, group=None, local_fn=None, grad=False):
    """Moment-matched mixture posterior over hyper samples (mcmc.py:84-93):
    mu = mean_i mu_i, s2 = mean_i (s2_i + (mu_i - mu)^2), samples split across
    the ranks.  `local_fn(hypers_slice, X) -> (mu_ (b, m), s2_ (b, m))`.
    grad=True also returns the input-gradients dmu = mean_i dmu_i and
    ds2 = mean_i (ds2_i + 2 (mu_i - mu)(dmu_i - dmu)); local_fn then returns
    (mu_, s2_, dmu_ (b, m, d), ds2_ (b, m, d)).  Two all-reduces either way:
    [sum mu_i, sum dmu_i], then the two centred sums."""
    rank, size = world(group)
    hypers = np.array(hypers, ndmin=2, dtype=float)
    X = np.array(X, ndmin=2, dtype=float)
    B, m, d = len(hypers), len(X), X.shape[1]
    lo, hi = shard_range(B, rank, size)
    if local_fn is None:
        if grad:
            from .meta.mcmc import _DeviceBatch
            local_fn = lambda h, x: _DeviceBatch(gp, h).predict(x, True)   # noqa: E731
        else:
            local_fn = lambda h, x: _batched('predict', gp, h, x)          # noqa: E731
    err = None
    parts = (np.empty((0, m)), np.empty((0, m))) + ((np.empty((0, m, d)), np.empty((0, m, d))) if grad else ())
    try:
        if hi > lo:
            parts = local_fn(hypers[lo:hi], X)
    except Exception as e:                # noqa: BLE001 -- e.g. LinAlgError on the one rank whose slice is non-PD
        err = e
    _raise_together(err, group)           # before the all-reduces: every rank raises, nobody deadlocks
    if not grad:
        mu_, s2_ = parts
        mu = all_reduce_sum(np.sum(mu_, axis=0), group)/B
        s2 = all_reduce_sum(np.sum(s2_ + (mu_ - mu)**2, axis=0), group)/B
        return mu, s2
    mu_, s2_, dmu_, ds2_ = (np.asarray(p, dtype=float) for p in parts)
    first = all_reduce_sum(np.concatenate([np.sum(mu_, axis=0), np.sum(dmu_, axis=0).ravel()]), group)/B
    mu, dmu = first[:m], first[m:].reshape(m, d)
    Mu = mu_ - mu
    second = all_reduce_sum(np.concatenate([np.sum(s2_ + Mu**2, axis=0),
                                            np.sum(ds2_ + 2*Mu[:, :, None]*(dmu_ - dmu), axis=0).ravel()]), group)/B
    return mu, second[:m], dmu, second[m:].reshape(m, d)
