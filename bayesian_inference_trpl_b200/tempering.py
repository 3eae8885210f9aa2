"""Parallel tempering of the ensemble sampler (ensemble.py): K copies ("rungs") of the stretch-move ensemble
sample lnL / T_t on a ladder T_0 < T_1 < ... < T_{K-1}, the hottest of which may be T = inf (the prior), and
neighbouring rungs exchange walkers after every step (include/trpl_b200_tempering.h, csrc/trpl_ensemble.cuh).
Hot rungs cross between separated modes and hand their states down to the cold rung; the per-rung mean lnL,
integrated over beta = 1/T, gives the log-evidence (thermodynamic integration, log_evidence).

Each half-step is one likelihood call over the moving half of every rung (K n rows), so the launch tail of
the fused solve is paid once for K ensembles.  Walker i of rung t only ever swaps with walker i of rung
t - 1, which keeps every swap on the rank that owns i: the chain does not depend on the number of ranks.
"""
import collections

import numpy as np
import torch

from . import _lib, distributed, engine, ensemble
from .ensemble import _host, _vp, _int, _i64, _u64, _u32, _dbl

MAX_RUNGS = 64                      # TRPL_MAX_RUNGS
TAG_SWAP = 3                        # TRPL_TAG_SWAP

# name -> (restype, argtypes) of every export, in the order of include/trpl_b200_tempering.h
_SIGNATURES = {
    "trpl_tempered_propose": (_int, [_vp, _i64, _i64, _i64, _i64, _int, _vp, _i64, _vp, _vp, _vp, _int, _int, _dbl,
                                     _u64, _u32, _vp, _i64, _vp, _int, _vp]),
    "trpl_tempered_accept": (_int, [_vp, _i64, _i64, _i64, _i64, _int, _vp, _int, _vp, _vp, _i64, _vp, _vp, _u64,
                                    _u32, _vp, _int, _vp]),
    "trpl_tempered_swap": (_int, [_vp, _i64, _i64, _i64, _i64, _int, _vp, _int, _vp, _u64, _u32, _vp, _int, _vp]),
}
EXPORTS = list(_SIGNATURES)

TemperedChain = collections.namedtuple("TemperedChain", "X lnl acceptance swap_acceptance temperatures")
TemperedChain.__doc__ = """X [steps+1, W, ncol] (engine units) of the cold rung only, lnl [steps+1, K, W] (the
log-likelihood as returned, NaN for a walker whose sample did not converge), acceptance [steps, K] (fraction of
each rung's W proposals accepted per step), swap_acceptance [steps, K-1] (fraction of the W walkers of rungs
t, t+1 exchanged per step, both halves), temperatures [K] (float64 numpy)."""

Evidence = collections.namedtuple("Evidence", "lnZ err mean_lnl extrapolated")
Evidence.__doc__ = """lnZ and its error estimate err, the mean lnL per rung [K], and whether the segment
[0, beta_min] was extrapolated (the hottest rung is finite)."""


def lib():
    """libtrpl_b200.so with the tempering entries bound."""
    L = ensemble.lib()
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(L, name)
        if fn.argtypes is None:
            fn.restype, fn.argtypes = restype, argtypes
    return L


def _call(name, dev, *args):
    return _lib.check(getattr(lib(), name)(*args, dev.index, engine._stream(dev)), name)


# ---- host logic ---------------------------------------------------------------------------------------------
def check_ladder(temperatures):
    """The ladder as float64, or ValueError: 1 <= K <= MAX_RUNGS entries, T_0 > 0, strictly increasing, and
    only the last entry may be inf (what the device entries enforce)."""
    T = np.array(temperatures, dtype=np.float64).reshape(-1)
    if not 1 <= T.shape[0] <= MAX_RUNGS:
        raise ValueError("a temperature ladder has 1 to %d rungs, got %d" % (MAX_RUNGS, T.shape[0]))
    with np.errstate(invalid="ignore"):
        ok = T[0] > 0 and bool((T[1:] > T[:-1]).all()) and not np.isinf(T[:-1]).any()
    if not ok:
        raise ValueError("temperatures must be strictly increasing from T_0 > 0, with only the last one "
                         "allowed to be inf; got %s" % list(T))
    return T


def geometric_ladder(K, t_max, prior_rung=True):
    """K temperatures: geometric from 1 to t_max (K - 1 of them when prior_rung, then T = inf)."""
    m = K - 1 if prior_rung else K
    if m < 1 or (m > 1 and not t_max > 1):
        raise ValueError("a geometric ladder needs at least one finite rung and t_max > 1")
    T = np.geomspace(1.0, t_max, m) if m > 1 else np.ones(1)
    return check_ladder(np.append(T, np.inf) if prior_rung else T)


def _trapezoid(beta, m):
    lnz = float(np.sum((beta[:-1] - beta[1:]) * (m[:-1] + m[1:]) / 2.0))
    return lnz + (beta[-1] * m[-1] if beta[-1] > 0 else 0.0)


def log_evidence(lnl, temperatures, burn):
    """Thermodynamic integration of lnl [steps+1, K, W] (TemperedChain.lnl): ln Z = integral over beta = 1/T
    from 0 to beta_0 of <lnL>_beta, with <lnL> the mean of the finite lnL of steps >= burn per rung, by the
    trapezoid rule over the ladder.  That is ln of the integral of prior x L^(1/T_0), the evidence when
    T_0 = 1.  When the hottest rung is finite, the segment [0, beta_min] is beta_min x <lnL>_hottest (as
    ptemcee does) and `extrapolated` is True.  err = |lnZ - the same rule on every other rung, both ends
    kept|: the discretisation error of the ladder, not the sampling error.  Returns an Evidence."""
    L = np.asarray(lnl.cpu() if isinstance(lnl, torch.Tensor) else lnl, dtype=np.float64)[burn:]
    beta = 1.0 / check_ladder(temperatures)
    if L.ndim != 3 or L.shape[1] != beta.shape[0]:
        raise ValueError("lnl must be [steps+1, K, W] with K = %d rungs" % beta.shape[0])
    fin = np.isfinite(L)
    with np.errstate(invalid="ignore", divide="ignore"):
        m = np.where(fin, L, 0.0).sum(axis=(0, 2)) / fin.sum(axis=(0, 2))
    lnz = _trapezoid(beta, m)
    every_other = sorted(set(range(0, beta.shape[0], 2)) | {beta.shape[0] - 1})
    err = abs(lnz - _trapezoid(beta[every_other], m[every_other]))
    return Evidence(lnz, err, m, bool(beta[-1] > 0))


# ---- device entries -----------------------------------------------------------------------------------------
def propose(X, first_walker, n_walkers, n_rungs, comp, minX, maxX, do_log, override_flags=0, a=2.0, seed=42,
            step=0, out=None):
    """Stretch proposals of the walkers X [K n, ncol] (row t n + i: walker first_walker + i of rung t, all in
    one half) against the complements comp [K ncol, W/2] (rung t's at rows t ncol ..).  Returns
    (Y [K n, ncol], logq [K n])."""
    dev = X.device
    assert X.dtype == torch.float64 and X.dim() == 2 and X.stride(1) == 1 and X.shape[0] % n_rungs == 0
    assert comp.device == dev and comp.dtype == torch.float64 and comp.stride(1) == 1
    rows, ncol = X.shape
    if comp.dim() != 2 or comp.shape[0] != n_rungs * ncol or comp.shape[1] < n_walkers // 2:
        raise ValueError("comp must hold every rung's complement, [%d rungs x %d columns, >= %d walkers], got %s"
                         % (n_rungs, ncol, n_walkers // 2, tuple(comp.shape)))
    lo, hi, dl = _host(minX, np.float64), _host(maxX, np.float64), _host(do_log, np.int32)
    if lo.shape[0] != ncol or hi.shape[0] != ncol or dl.shape[0] != ncol:
        raise ValueError("one bound and one do_log flag per column of X are required")
    Y = out if out is not None else torch.empty((rows, ncol), dtype=torch.float64, device=dev)
    logq = torch.empty(rows, dtype=torch.float64, device=dev)
    if rows == 0:                                       # an empty tensor has no data pointer
        return Y, logq
    _call("trpl_tempered_propose", dev, engine._ptr(X), rows // n_rungs, engine._row_stride(X), int(first_walker),
          int(n_walkers), int(n_rungs), engine._ptr(comp), comp.stride(0) if comp.shape[0] > 1 else comp.shape[1],
          lo.ctypes.data_as(_vp), hi.ctypes.data_as(_vp), dl.ctypes.data_as(_vp), ncol, int(override_flags),
          float(a), int(seed), int(step), engine._ptr(Y), engine._row_stride(Y), engine._ptr(logq))
    return Y, logq


def accept_(X, lnl, Y, lnl_y, logq, first_walker, n_walkers, temperatures, seed=42, step=0, accepted=None):
    """Accept/reject in place, rung t at temperatures[t]: accepted rows of Y replace those of X [K n, ncol],
    their lnL that of lnl [K n].  Returns the int32 accepted flags [K n]."""
    dev = X.device
    T = check_ladder(temperatures)
    rows, ncol = X.shape
    assert lnl.shape == (rows,) and lnl_y.shape == (rows,) and logq.shape == (rows,) and Y.shape[0] == rows
    assert all(t.is_contiguous() for t in (lnl, lnl_y, logq)) and Y.stride(1) == 1 and X.stride(1) == 1
    assert rows % T.shape[0] == 0
    acc = accepted if accepted is not None else torch.empty(rows, dtype=torch.int32, device=dev)
    if rows == 0:
        return acc
    _call("trpl_tempered_accept", dev, engine._ptr(X), rows // T.shape[0], engine._row_stride(X),
          int(first_walker), int(n_walkers), T.shape[0], T.ctypes.data_as(_vp), ncol, engine._ptr(lnl),
          engine._ptr(Y), engine._row_stride(Y), engine._ptr(lnl_y), engine._ptr(logq), int(seed), int(step),
          engine._ptr(acc))
    return acc


def swap_(X, lnl, first_walker, n_walkers, temperatures, seed=42, step=0, swapped=None):
    """Replica exchange in place between neighbouring rungs of X [K n, ncol] and lnl [K n], hottest pair
    first.  Returns the int32 swap flags [(K-1) n] (entry (t-1) n + i: walker i between rungs t-1 and t)."""
    dev = X.device
    T = check_ladder(temperatures)
    K = T.shape[0]
    rows, ncol = X.shape
    assert lnl.shape == (rows,) and lnl.is_contiguous() and X.stride(1) == 1 and rows % K == 0
    n = rows // K
    sw = swapped if swapped is not None else torch.empty((K - 1) * n, dtype=torch.int32, device=dev)
    if rows == 0:
        return sw
    _call("trpl_tempered_swap", dev, engine._ptr(X), n, engine._row_stride(X), int(first_walker), int(n_walkers),
          K, T.ctypes.data_as(_vp), ncol, engine._ptr(lnl), int(seed), int(step),
          engine._ptr(sw) if sw.numel() else None)
    return sw


# ---- driver -------------------------------------------------------------------------------------------------
def initial_walkers(n_walkers, n_rungs, minX, maxX, do_log, seed, override_flags=0, rank=0, world=1,
                    device=None):
    """This rank's initial walkers [K (nA + nB), ncol], rung-major, each rung in ensemble.local_rows order:
    rung t takes rows [t W, (t+1) W) of the global engine.random_grid_device draw under `seed`, so rung 0
    equals ensemble.initial_walkers.  A rank may hold no walkers of a half (more ranks than W/2)."""
    dev = engine.require_cuda(device)
    ncol = len(minX)
    parts = [engine.random_grid_device(minX, maxX, do_log, hi - lo, seed, first_sample=t * n_walkers + lo,
                                       override_flags=override_flags, device=dev.index)
             if hi > lo else torch.empty((0, ncol), dtype=torch.float64, device=dev)     # no data pointer to fill
             for t in range(n_rungs) for lo, hi in ensemble.local_rows(n_walkers, rank, world)]
    return torch.cat(parts)


def _gather(ex, local, h):
    """ex.gather_rows of [rows, n] shards.  Collective: a rank whose shard is empty (n = 0) still takes part.
    Only a table without rows (steps = 0, or the swap flags of one rung), the same on every rank, is skipped."""
    if local.shape[0] == 0:
        return local.new_empty((0, h))
    return ex.gather_rows(local.contiguous(), h)


def sample(X0, log_likelihood, minX, maxX, do_log, steps, temperatures, n_walkers=None, override_flags=0, a=2.0,
           seed=42, exchange=None, timer=None):
    """Run `steps` steps of the tempered ensemble whose local walkers are the device tensor X0
    [K (nA + nB), ncol] (initial_walkers order; with one rank, K whole ensembles of W walkers), in engine
    units, on the ladder `temperatures` (K entries, see check_ladder).

    The contract is that of ensemble.sample: `log_likelihood(X [m, ncol]) -> lnL [m]`, the `exchange`
    object, `timer`.  A half-step gathers the other half of every rung with one gather_rows, proposes,
    evaluates the K n rows of the moving half with ONE log_likelihood call and accepts; after both halves,
    each half's walkers swap between neighbouring rungs.  Returns a TemperedChain, complete on every rank."""
    ex = exchange if exchange is not None else distributed.TorchExchange()
    rank, world = ex.rank_world()
    T = check_ladder(temperatures)
    K = T.shape[0]
    dev = X0.device
    ncol = X0.shape[1]
    W = int(n_walkers if n_walkers is not None else X0.shape[0] // K)
    ensemble.check_walkers(W, int(ensemble.free_columns(minX, maxX, override_flags).sum()))
    h = W // 2
    rows = ensemble.local_rows(W, rank, world)
    nA, nB = rows[0][1] - rows[0][0], rows[1][1] - rows[1][0]
    if X0.shape != (K * (nA + nB), ncol):
        raise ValueError("rank %d of %d holds %d walkers of half A and %d of half B in each of %d rungs, X0 has "
                         "%d rows" % (rank, world, nA, nB, K, X0.shape[0]))
    X = X0.to(torch.float64).reshape(K, nA + nB, ncol)
    halves = [X[:, sl].clone(memory_format=torch.contiguous_format).reshape(K * n, ncol)     # copies of X0
              for sl, n in ((slice(0, nA), nA), (slice(nA, None), nB))]
    sizes = (nA, nB)
    lnl = [torch.empty(K * n, dtype=torch.float64, device=dev) for n in sizes]
    if timer is not None:
        timer("solve")
    if nA + nB:
        first = log_likelihood(torch.cat(halves))
        lnl[0].copy_(first[:K * nA])
        lnl[1].copy_(first[K * nA:])
    if timer is not None:
        timer("other")
    chain_x = torch.empty((steps + 1, nA + nB, ncol), dtype=torch.float64, device=dev)
    chain_l = torch.empty((steps + 1, K, nA + nB), dtype=torch.float64, device=dev)
    chain_a = torch.empty((steps, K, nA + nB), dtype=torch.float64, device=dev)
    chain_s = torch.empty((steps, K - 1, nA + nB), dtype=torch.float64, device=dev)
    acc = [torch.empty(K * n, dtype=torch.int32, device=dev) for n in sizes]
    swp = [torch.empty((K - 1) * n, dtype=torch.int32, device=dev) for n in sizes]

    def record(s):
        for k, (n, sl) in enumerate(zip(sizes, (slice(0, nA), slice(nA, nA + nB)))):
            chain_x[s, sl] = halves[k][:n]                      # rung 0 only
            chain_l[s, :, sl] = lnl[k].view(K, n)

    record(0)
    for step in range(steps):
        for k in range(2):
            n, other, n_other = sizes[k], halves[1 - k], sizes[1 - k]
            comp = _gather(ex, other.view(K, n_other, ncol).permute(0, 2, 1).reshape(K * ncol, n_other), h)
            Y, logq = propose(halves[k], rows[k][0], W, K, comp, minX, maxX, do_log, override_flags, a, seed, step)
            if timer is not None:
                timer("solve")
            lnl_y = log_likelihood(Y) if Y.shape[0] else torch.empty(0, dtype=torch.float64, device=dev)
            if timer is not None:
                timer("other")
            accept_(halves[k], lnl[k], Y, lnl_y, logq, rows[k][0], W, T, seed, step, accepted=acc[k])
        for k in range(2):
            swap_(halves[k], lnl[k], rows[k][0], W, T, seed, step, swapped=swp[k])
        record(step + 1)
        chain_a[step] = torch.cat([a.view(K, n) for a, n in zip(acc, sizes)], dim=1)
        chain_s[step] = torch.cat([s.view(K - 1, n) for s, n in zip(swp, sizes)], dim=1)
    full_x, full_l, full_a, full_s = [], [], [], []
    for k, sl in enumerate((slice(0, nA), slice(nA, nA + nB))):
        n = sl.stop - sl.start
        xs = chain_x[:, sl].permute(0, 2, 1).reshape((steps + 1) * ncol, n)
        full_x.append(_gather(ex, xs, h).reshape(steps + 1, ncol, h).permute(0, 2, 1))
        full_l.append(_gather(ex, chain_l[:, :, sl].reshape((steps + 1) * K, n), h).reshape(steps + 1, K, h))
        full_a.append(_gather(ex, chain_a[:, :, sl].reshape(steps * K, n), h).reshape(steps, K, h))
        full_s.append(_gather(ex, chain_s[:, :, sl].reshape(steps * (K - 1), n), h).reshape(steps, K - 1, h))
    return TemperedChain(torch.cat(full_x, dim=1).contiguous(), torch.cat(full_l, dim=2).contiguous(),
                         torch.cat(full_a, dim=2).mean(dim=2),
                         torch.cat(full_s, dim=2).mean(dim=2), T)
