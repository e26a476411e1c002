"""
Batched GP work on independent light curves / kernels, and its sharding across GPUs.

The reference has no batch interface (it loops a Python ``GaussianProcess`` per star:
notebooks/paper/runtime-speed.ipynb:40-42); these helpers are the same calls
(``compute`` + ``log_likelihood``, ``compute`` + ``sample``, ``kernel.get_psd``) issued for
B independent units at once through the fused CUDA kernels, which materialise nothing of
size N*J.  Units are independent, so multi-GPU is pure sharding: rank r owns a contiguous
block of units (balanced by N*J^2), and the only collective is the final gather of the
per-unit scalars (SURVEY.md section 8e).
"""
import numpy as np

from .solver import Geometry, KernelBatch, default_solver

__all__ = ['log_likelihood', 'log_likelihood_gradient', 'sample', 'shard_bounds', 'shard', 'gather_concat']

_LOG_2PI = float(np.log(2 * np.pi))


def _as_batch(kernels):
    return kernels if isinstance(kernels, KernelBatch) else KernelBatch(kernels)


def _geometry(kb, t, lengths):
    if lengths is None:
        t = np.asarray(t) if not hasattr(t, 'data_ptr') else t
        if hasattr(t, 'data_ptr') or t.ndim == 1:
            N = t.numel() if hasattr(t, 'data_ptr') else t.shape[0]
            return Geometry.shared_t(kb.B, int(N))
        assert t.shape[0] == kb.B
        return Geometry.ragged([t.shape[1]] * kb.B)
    return Geometry.ragged(lengths)


class PendingLogLikelihood:
    """Result of ``log_likelihood(..., wait=False)``: the copies and the kernel are queued; ``result()``
    blocks until THIS call has completed (not later ones) and returns what ``log_likelihood`` returns."""

    def __init__(self, solver, ticket, finish):
        self._solver, self._ticket, self._finish, self._value = solver, ticket, finish, None

    def result(self):
        if self._finish is not None:
            self._solver.wait(self._ticket)
            self._value, self._finish = self._finish(), None
        return self._value


def log_likelihood(kernels, t, y, diag=None, lengths=None, mean=0.0, quiet=True, solver=None,
                   return_parts=False, flags=0, wait=True):
    """log-likelihood of B light curves under B kernels.

    ``t``: ``[N]`` (one cadence shared by all units), ``[B, N]``, or a flat concatenation
    with ``lengths``;  ``y``, ``diag``: ``[B, N]`` or flat -- or, with
    ``flags=solver.FLAG_SHARED_Y``, laid out like ``t`` (one light curve for many
    hyper-parameter sets: nothing is replicated).  Non-positive-definite units give
    ``-inf`` (``quiet=True``) or raise ``LinAlgError``."""
    from .solver import LinAlgError
    kb = _as_batch(kernels)
    geom = _geometry(kb, t, lengths)
    solver = solver or default_solver()
    if not hasattr(y, 'data_ptr'):
        y = np.ascontiguousarray(y, dtype=np.float64)
        if np.any(mean != 0.0):
            y = y - mean
    from .solver import FLAG_ASYNC
    logdet, quad, status = solver.loglike(kb, geom, t, y, diag, flags=flags | (0 if wait else FLAG_ASYNC))

    def finish():
        N = np.diff(geom.n_off)
        ll = -0.5 * (quad + logdet + N * _LOG_2PI)
        bad = status != 0
        if np.any(bad):
            if not quiet:
                b = int(np.flatnonzero(bad)[0])
                raise LinAlgError(f"unit {b}: failed to factorize, d[{status[b] - 1}] <= 0")
            ll = np.where(bad, -np.inf, ll)
        if return_parts:
            return ll, logdet, quad, status
        return ll

    if not wait:
        # (``wait=False``: y / t must stay alive and unchanged until result(); the next call's copies
        # and kernels can be queued behind this one -- bench.py's end-to-end loop)
        return PendingLogLikelihood(solver, solver.ticket(), finish)
    return finish()


def log_likelihood_gradient(S0, w0, Q, delta, t, y, diag=None, wrt=('S0', 'w0', 'Q'), rel_step=2e-3,
                            solver=None, return_value=False):
    """Gradient of log L with respect to the SHO hyper-parameters of every term, ``d logL / d ln p``
    for p in (S0_j, w0_j, Q_j) -- what a fit of the kernel to a light curve needs (the reference fits
    with celerite2.jax + BFGS: notebooks/virgo_lc.ipynb:48; SURVEY.md 8f-4).

    Method: NOT an adjoint sweep.  The fused log-likelihood kernel runs one sequence per SM, so a
    single light curve leaves 147 of 148 SMs idle; here every hyper-parameter gets four perturbed
    kernels (p (1 +- h), p (1 +- 2h): fourth-order central differences in ln p) and all 4 P + 1
    kernels are scanned in ONE batched launch against the one light curve (``FLAG_SHARED_Y``: y is
    passed once).  For the solar kernel's 258 parameters that is 1033 sequences = 7 waves of 148, the
    wall time of ~7 single log-likelihoods -- what an O(N J^2) adjoint pass on one SM would cost too.
    Steps: ``rel_step`` in ln p, except ln w0 of a resonant term, where log L varies on the scale
    of the line width 1 / Q: h = min(rel_step, 0.05 / Q_j).  Accuracy: truncation ~h^4, rounding
    ~1e-12 |log L| / h: ~1e-6 of the gradient's norm (tests/test_gpu_parity.py checks it against a
    longdouble evaluation of the kernel definition).  Returns ``grad[len(wrt), J/2]`` (and log L at the centre with ``return_value``)."""
    from .feeder import HyperparameterBatch, kernel_batch_from_sho
    from .solver import FLAG_SHARED_Y
    S0, w0, Q = (np.ascontiguousarray(v, dtype=np.float64) for v in (S0, w0, Q))
    nt = len(S0)
    names = list(wrt)
    P = len(names) * nt
    stencil = np.array([-2.0, -1.0, 1.0, 2.0])
    h = np.full((len(names), nt), float(rel_step))
    for i, name in enumerate(names):
        if name == 'w0':
            h[i] = np.minimum(rel_step, 0.05 / np.maximum(Q, 0.5))
    rows = 4 * P + 1
    par = {'S0': np.tile(S0, (rows, 1)), 'w0': np.tile(w0, (rows, 1)), 'Q': np.tile(Q, (rows, 1))}
    for i, name in enumerate(names):
        for j in range(nt):
            r0 = 1 + 4 * (i * nt + j)
            par[name][r0:r0 + 4, j] *= np.exp(stencil * h[i, j])
    hpb = HyperparameterBatch(par['S0'].ravel(), par['w0'].ravel(), par['Q'].ravel(),
                              np.arange(rows + 1, dtype=np.int64) * nt)
    kb = kernel_batch_from_sho(hpb, delta)
    solver = solver or default_solver()
    ll = log_likelihood(kb, t, y, diag, solver=solver, flags=FLAG_SHARED_Y)
    f = ll[1:].reshape(P, 4)
    grad = (f[:, 0] - 8 * f[:, 1] + 8 * f[:, 2] - f[:, 3]) / (12 * h.ravel())
    grad = grad.reshape(len(names), nt)
    return (grad, float(ll[0])) if return_value else grad


def sample(kernels, t, diag=None, lengths=None, normals=None, seed=0, seq0=0, solver=None,
           subtract_mean=True, out=None, flags=0, size=None):
    """One GP draw per unit: ``x = L (sqrt(d) o n)``.  ``normals=None`` draws n on the device
    from Philox4x32-10 keyed by ``seed`` and the global unit index ``seq0 + b``
    (reproducible on the host with :mod:`gadfly_b200.philox`).  ``subtract_mean`` applies the
    reference's mean subtraction (gadfly/gp.py:392): over the draw's samples for one draw, over the
    realisations at each time stamp for ``size`` of them.  It needs the draws on the host, so it
    cannot be combined with ``FLAG_ASYNC`` (the buffer is written after this returns)."""
    from .solver import FLAG_ASYNC
    if subtract_mean and (flags & FLAG_ASYNC):
        raise ValueError("subtract_mean needs the draws: pass subtract_mean=False with FLAG_ASYNC")
    kb = _as_batch(kernels)
    geom = _geometry(kb, t, lengths)
    solver = solver or default_solver()
    if size is not None:
        # ``size`` realisations per unit on ONE factor (celerite2's sample(size=k), reference
        # gadfly/gp.py:372-395): returns [B, size, N] (or a list of [size, N_b]), Philox realisation
        # index seq0 + b size + r
        k = int(size)
        x, logdet, status = solver.sample_multi(kb, geom, t, k, diag, normals, seed=seed, seq0=seq0, out=out,
                                                flags=flags)
        if hasattr(x, 'data_ptr'):
            return x, status
        rows = [x[k * geom.n_off[b]:k * geom.n_off[b + 1]].reshape(k, -1) for b in range(kb.B)]
        if subtract_mean:
            # celerite2's sample(size=k) returns [k, N]; the reference subtracts result.mean(axis=0)
            for r in rows:
                if r.size:
                    r -= r.mean(axis=0, keepdims=True)
        return (np.stack(rows) if lengths is None else rows), status
    x, logdet, status = solver.sample(kb, geom, t, diag, normals, seed=seed, seq0=seq0, out=out,
                                      flags=flags)
    if hasattr(x, 'data_ptr'):
        return x, status
    rows = [x[geom.n_off[b]:geom.n_off[b + 1]] for b in range(kb.B)]
    if subtract_mean:
        for r in rows:
            if len(r):
                r -= r.mean()
    if lengths is None:
        return x.reshape(kb.B, -1), status
    return rows, status


# ---- sharding -------------------------------------------------------------------------
def shard_bounds(cost, world):
    """Contiguous block boundaries [world+1] that balance ``sum(cost)`` per rank."""
    cost = np.asarray(cost, dtype=np.float64)
    B = len(cost)
    if B == 0:
        return np.zeros(world + 1, dtype=np.int64)
    csum = np.concatenate([[0.0], np.cumsum(cost)])
    targets = csum[-1] * np.arange(1, world) / world
    cuts = np.searchsorted(csum, targets, side='left')
    # pick the closer of the two neighbouring cut points
    cuts = np.where((cuts > 0) & (np.abs(csum[np.maximum(cuts - 1, 0)] - targets)
                                  < np.abs(csum[np.minimum(cuts, B)] - targets)), cuts - 1, cuts)
    bounds = np.concatenate([[0], np.clip(cuts, 0, B), [B]]).astype(np.int64)
    return np.maximum.accumulate(bounds)


def shard(B, rank, world, cost=None):
    """Index range [lo, hi) of the units rank ``rank`` owns."""
    if cost is None:
        cost = np.ones(B)
    b = shard_bounds(cost, world)
    return int(b[rank]), int(b[rank + 1])


def gather_concat(local, bounds=None, group=None):
    """All-gather per-unit results (1-D arrays of per-rank length) into the full array on every rank:
    the only collective of the path (SURVEY.md section 8e).  ``local`` is a numpy array or a torch
    tensor; a CUDA tensor stays on the device and is gathered by NCCL on torch's current stream (the
    result is a CUDA tensor), anything else goes through the process group's backend and comes back
    as numpy.  ``bounds`` [world + 1] are the shard boundaries (:func:`shard_bounds`): every rank
    knows them, so no sizes are exchanged; without them one extra all-gather of the lengths is made."""
    import torch
    import torch.distributed as dist
    is_tensor = hasattr(local, 'data_ptr')
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local if is_tensor else np.asarray(local)
    world = dist.get_world_size(group)
    backend = dist.get_backend(group)
    if is_tensor and local.is_cuda:
        x = local.contiguous()
    else:
        dev = torch.device('cuda', torch.cuda.current_device()) if backend == 'nccl' else torch.device('cpu')
        x = torch.as_tensor(np.ascontiguousarray(local.cpu().numpy() if is_tensor else local)).to(dev)
    if bounds is not None:
        sizes = [int(v) for v in np.diff(np.asarray(bounds, dtype=np.int64))]
        assert len(sizes) == world and sizes[dist.get_rank(group)] == x.numel(), "bounds do not match the shard"
    else:
        mine = torch.tensor([x.numel()], dtype=torch.int64, device=x.device)
        every = torch.empty(world, dtype=torch.int64, device=x.device)
        dist.all_gather_into_tensor(every, mine, group=group)
        sizes = every.tolist()
    m = max(sizes) if sizes else 0
    if m == 0:
        out = x.new_empty(0)
    else:
        pad = x if x.numel() == m else torch.cat([x, x.new_zeros(m - x.numel())])
        flat = x.new_empty(world * m)
        dist.all_gather_into_tensor(flat, pad, group=group)
        out = flat if all(sz == m for sz in sizes) else torch.cat([flat[r * m:r * m + sz] for r, sz in enumerate(sizes)])
    if is_tensor and local.is_cuda:
        return out
    return out.cpu().numpy()
