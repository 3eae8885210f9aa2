"""Affine-invariant ensemble MCMC (the stretch move of Goodman & Weare 2010, in emcee's two-half form,
Foreman-Mackey et al. 2013) around the fused likelihood: proposals and accept/reject run on the device
(include/trpl_b200_ensemble.h, csrc/trpl_ensemble.cuh), each half-step is one likelihood call of the
half's walkers, and the walkers of each half are sharded over ranks by `distributed.shard_bounds`.

The target is lnL / temperature on the prior box, in the prior's coordinates (log10 for do_log columns),
where the prior is uniform.  Randomness is counter-based (seed, walker, step), so the chain does not depend
on the number of ranks.
"""
import collections
import ctypes

import numpy as np
import torch

from . import _lib, distributed, engine

_vp, _int, _i64, _u64, _u32, _dbl = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64,
                                     ctypes.c_uint32, ctypes.c_double)

# name -> (restype, argtypes) of every export, in the order of include/trpl_b200_ensemble.h
_SIGNATURES = {
    "trpl_stretch_propose": (_int, [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _int, _int, _dbl, _u64,
                                    _u32, _vp, _i64, _vp, _int, _vp]),
    "trpl_stretch_accept": (_int, [_vp, _i64, _i64, _i64, _i64, _int, _vp, _vp, _i64, _vp, _vp, _dbl, _u64, _u32,
                                   _vp, _int, _vp]),
}
EXPORTS = list(_SIGNATURES)

Chain = collections.namedtuple("Chain", "X lnl acceptance")
Chain.__doc__ = """X [steps+1, W, ncol] (engine units), lnl [steps+1, W] (the log-likelihood as returned, NaN for a
walker whose sample did not converge), acceptance [steps] (fraction of the W proposals accepted per step)."""


def lib():
    """libtrpl_b200.so with the ensemble entries bound."""
    L = _lib.lib()
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(L, name)
        if fn.argtypes is None:
            fn.restype, fn.argtypes = restype, argtypes
    return L


def _call(name, dev, *args):
    return _lib.check(getattr(lib(), name)(*args, dev.index, engine._stream(dev)), name)


def _host(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


# ---- host logic ---------------------------------------------------------------------------------------------
def override_sources(override_flags, ncol):
    """{target column: source column} of the override flags (bit 0: 2 <- 3, bit 1: 6 <- 5, bit 2: 8 <- 7)."""
    pairs = ((1, 2, 3, 3), (2, 6, 5, 6), (4, 8, 7, 8))
    return {t: s for bit, t, s, need in pairs if override_flags & bit and ncol > need}


def free_columns(minX, maxX, override_flags=0):
    """Mask of the columns the sampler moves: not fixed (minX == maxX) and not an override target."""
    lo, hi = np.asarray(minX, dtype=np.float64), np.asarray(maxX, dtype=np.float64)
    free = lo != hi
    for t in override_sources(override_flags, lo.shape[0]):
        free[t] = False
    return free


def check_walkers(n_walkers, d):
    """W must be even and at least 2 max(d, 1) for d free columns (what the device entries enforce)."""
    if n_walkers % 2 or n_walkers < 2 * max(d, 1):
        raise ValueError("the ensemble needs an even number of walkers >= 2 x %d free parameters, got %d"
                         % (max(d, 1), n_walkers))


def local_rows(n_walkers, rank, world):
    """This rank's walkers: global ranges [(lo, hi) in half A, (lo, hi) in half B], the shard_bounds slice of
    each half.  The rank holds them in that order (A rows, then B rows)."""
    h = n_walkers // 2
    lo, hi = distributed.shard_bounds(h, rank, world)
    return [(lo, hi), (h + lo, h + hi)]


# ---- device entries -----------------------------------------------------------------------------------------
def propose(X, first_walker, n_walkers, comp, minX, maxX, do_log, override_flags=0, a=2.0, seed=42, step=0,
            out=None):
    """Stretch proposals of the walkers X [n, ncol] (global indices first_walker + i, all in one half) against
    the complement comp [ncol, W/2] (the other half, transposed).  Returns (Y [n, ncol], logq [n])."""
    dev = X.device
    assert X.dtype == torch.float64 and X.dim() == 2 and X.stride(1) == 1
    assert comp.device == dev and comp.dtype == torch.float64 and comp.stride(1) == 1
    n, ncol = X.shape
    lo, hi, dl = _host(minX, np.float64), _host(maxX, np.float64), _host(do_log, np.int32)
    if lo.shape[0] != ncol or hi.shape[0] != ncol or dl.shape[0] != ncol:
        raise ValueError("one bound and one do_log flag per column of X are required")
    Y = out if out is not None else torch.empty((n, ncol), dtype=torch.float64, device=dev)
    logq = torch.empty(n, dtype=torch.float64, device=dev)
    if n == 0:                                          # an empty tensor has no data pointer
        return Y, logq
    _call("trpl_stretch_propose", dev, engine._ptr(X), n, engine._row_stride(X), int(first_walker), int(n_walkers),
          engine._ptr(comp), comp.stride(0) if comp.shape[0] > 1 else comp.shape[1],
          lo.ctypes.data_as(_vp), hi.ctypes.data_as(_vp), dl.ctypes.data_as(_vp), ncol, int(override_flags),
          float(a), int(seed), int(step), engine._ptr(Y), engine._row_stride(Y), engine._ptr(logq))
    return Y, logq


def accept_(X, lnl, Y, lnl_y, logq, first_walker, n_walkers, temperature=1.0, seed=42, step=0, accepted=None):
    """Accept/reject in place: accepted rows of Y replace those of X, their lnL that of lnl.  Returns the
    int32 accepted flags [n]."""
    dev = X.device
    n, ncol = X.shape
    assert lnl.shape == (n,) and lnl_y.shape == (n,) and logq.shape == (n,) and Y.shape[0] == n
    assert all(t.is_contiguous() for t in (lnl, lnl_y, logq)) and Y.stride(1) == 1 and X.stride(1) == 1
    acc = accepted if accepted is not None else torch.empty(n, dtype=torch.int32, device=dev)
    if n == 0:
        return acc
    _call("trpl_stretch_accept", dev, engine._ptr(X), n, engine._row_stride(X), int(first_walker), int(n_walkers),
          ncol, engine._ptr(lnl), engine._ptr(Y), engine._row_stride(Y), engine._ptr(lnl_y), engine._ptr(logq),
          float(temperature), int(seed), int(step), engine._ptr(acc))
    return acc


# ---- driver -------------------------------------------------------------------------------------------------
def solver_loglik(problem, log_pl=True, self_normalize=False, emulate_f32=False):
    """log_likelihood(X rows) -> lnL [n] of the one observation file of `problem` through engine.solve_loglik."""
    if problem.E != 1:
        raise ValueError("one ensemble samples the posterior of one observation file; got %d" % problem.E)

    def log_likelihood(X):
        lnl, _, _ = engine.solve_loglik(X, problem, log_pl=log_pl, self_normalize=self_normalize,
                                        emulate_f32=emulate_f32)
        return lnl[0]
    return log_likelihood


def initial_walkers(n_walkers, minX, maxX, do_log, seed, override_flags=0, rank=0, world=1, device=None):
    """This rank's initial walkers (local_rows order) drawn from the prior on the device with
    engine.random_grid_device: the rows of the global draw of n_walkers samples under `seed`."""
    parts = [engine.random_grid_device(minX, maxX, do_log, hi - lo, seed, first_sample=lo,
                                       override_flags=override_flags, device=device)
             for lo, hi in local_rows(n_walkers, rank, world)]
    return torch.cat(parts)


def sample(X0, log_likelihood, minX, maxX, do_log, steps, n_walkers=None, override_flags=0, temperature=1.0,
           a=2.0, seed=42, exchange=None, timer=None):
    """Run `steps` stretch-move steps of the ensemble whose local walkers (local_rows order; with one rank, the
    whole ensemble [W, ncol]) are the device tensor X0, in engine units.

    `log_likelihood(X [n, ncol]) -> lnL [n]` (float64, on X's device) evaluates the walkers, e.g.
    solver_loglik(problem).  Every half-step gathers the complement half through `exchange`
    (distributed.TorchExchange by default, or an nccl.Communicator) and evaluates this rank's walkers of the
    moving half.  `timer(tag)`, if given, is called with "solve" before and "other" after each likelihood
    call, the initial one included (for measurements).  Returns a Chain, complete on every rank."""
    ex = exchange if exchange is not None else distributed.TorchExchange()
    rank, world = ex.rank_world()
    dev = X0.device
    ncol = X0.shape[1]
    W = int(n_walkers if n_walkers is not None else X0.shape[0])
    check_walkers(W, int(free_columns(minX, maxX, override_flags).sum()))
    if not temperature > 0:
        raise ValueError("temperature must be > 0")
    h = W // 2
    rows = local_rows(W, rank, world)
    nA, nB = rows[0][1] - rows[0][0], rows[1][1] - rows[1][0]
    if X0.shape != (nA + nB, ncol):
        raise ValueError("rank %d of %d holds %d walkers of half A and %d of half B, X0 has %d rows"
                         % (rank, world, nA, nB, X0.shape[0]))
    X = X0.to(torch.float64).contiguous().clone()
    halves = [(X[:nA], slice(0, nA)), (X[nA:], slice(nA, nA + nB))]
    lnl = torch.empty(nA + nB, dtype=torch.float64, device=dev)
    if timer is not None:
        timer("solve")
    if nA + nB:
        lnl.copy_(log_likelihood(X))
    if timer is not None:
        timer("other")
    chain_x = torch.empty((steps + 1, nA + nB, ncol), dtype=torch.float64, device=dev)
    chain_l = torch.empty((steps + 1, nA + nB), dtype=torch.float64, device=dev)
    chain_a = torch.empty((steps, nA + nB), dtype=torch.float64, device=dev)
    acc = torch.empty(nA + nB, dtype=torch.int32, device=dev)
    chain_x[0] = X
    chain_l[0] = lnl
    for step in range(steps):
        for k, (Xk, sl) in enumerate(halves):
            other = halves[1 - k][0]
            comp = ex.gather_rows(other.t().contiguous(), h)              # [ncol, W/2] on every rank
            first = rows[k][0]
            Y, logq = propose(Xk, first, W, comp, minX, maxX, do_log, override_flags, a, seed, step)
            if timer is not None:
                timer("solve")
            lnl_y = log_likelihood(Y) if Y.shape[0] else torch.empty(0, dtype=torch.float64, device=dev)
            if timer is not None:
                timer("other")
            accept_(Xk, lnl[sl], Y, lnl_y, logq, first, W, temperature, seed, step, accepted=acc[sl])
        chain_x[step + 1] = X
        chain_l[step + 1] = lnl
        chain_a[step] = acc
    full_x, full_l, full_a = [], [], []
    for k, (_, sl) in enumerate(halves):
        n = sl.stop - sl.start
        xs = chain_x[:, sl].permute(0, 2, 1).reshape((steps + 1) * ncol, n)
        full_x.append(ex.gather_rows(xs.contiguous(), h).reshape(steps + 1, ncol, h).permute(0, 2, 1))
        full_l.append(ex.gather_rows(chain_l[:, sl].contiguous(), h))
        full_a.append(ex.gather_rows(chain_a[:, sl].contiguous(), h))
    acceptance = torch.cat(full_a, dim=1).mean(dim=1) if steps else torch.empty(0, dtype=torch.float64, device=dev)
    return Chain(torch.cat(full_x, dim=1).contiguous(), torch.cat(full_l, dim=1).contiguous(), acceptance)
