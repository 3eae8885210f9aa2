"""Host-side mirror of the reference driver `bayeslib.py` (random_grid :18-32, make_grid :34-76,
simulate :83-205, bayes :207-252): same function names, argument order and in-place outputs, so
code written against the reference keeps working.  Two ways through `simulate`:

  * fused (default, gpu_info["fused"] != False): every sample of this rank goes through ONE
    trpl_solve_loglik launch -- forward model, optional self-normalisation, log10, time
    interpolation and squared-residual sum stay on the B200; only lnL comes back;
  * staged (gpu_info["fused"] = False): the reference's own sequence of calls
    model() -> fastlog() -> host interpolation -> prob(), block by block, with the float32 PL
    buffer of bayeslib.py:137 -- bit-compatible with the reference pipeline, and as slow.
"""
import os
import sys
import time

import numpy as np
import torch

from . import engine
from .probs import fastlog, prob


def random_grid(minX, maxX, do_log, num_points, do_grid=False, refs=None):
    """Uniform (or log-uniform) draws inside [minX, maxX]; one numpy RNG call per free parameter,
    in column order, so a seeded run reproduces the reference's sample matrix bit for bit."""
    lo = np.asarray(minX, dtype=np.float64)
    hi = np.asarray(maxX, dtype=np.float64)
    X = np.empty((num_points, lo.shape[0]))
    for j in range(lo.shape[0]):
        if lo[j] == hi[j]:
            X[:, j] = lo[j]
            continue
        if do_log[j]:
            X[:, j] = 10 ** np.random.uniform(np.log10(lo[j]), np.log10(hi[j]), (num_points,))
        else:
            X[:, j] = np.random.uniform(lo[j], hi[j], (num_points,))
    return X


def make_grid(N, P, num_exp, minX, maxX, do_log, sim_flags, nref=None, minP=None, refs=None):
    """Sample matrix X [S,13], zeroed likelihood table P [num_exp,S] and sample ids N."""
    if not sim_flags["random_sample"]:
        raise NotImplementedError("the deprecated coarse-grid sampler (Legacy/legacy.py) is not "
                                  "part of the B200 engine; use random_sample=True")
    S = sim_flags["num_points"]
    N = np.arange(S)
    X = random_grid(minX, maxX, do_log, S, refs=refs)
    P = np.zeros((num_exp, S))
    if sim_flags["override_equal_mu"]:
        X[:, 2] = X[:, 3]
    if sim_flags["override_equal_s"]:
        X[:, 6] = X[:, 5]
    if sim_flags["override_equal_auger"]:
        X[:, 8] = X[:, 7]
    return N, P, X


def almost_equal(x, x0, threshold=1e-10):
    if x.shape != x0.shape:
        return False
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.abs(np.nanmax((x - x0) / x0)) < threshold


def interpolate_rows(sim_times, rows, times):
    """Linear interpolation of every row onto `times` with the bracketing rule scipy's griddata /
    interp1d applies to 1-D data (bayeslib.py:186-189), vectorised over samples."""
    hi = np.clip(np.searchsorted(sim_times, times), 1, len(sim_times) - 1)
    lo = hi - 1
    span = sim_times[hi] - sim_times[lo]
    with np.errstate(invalid="ignore"):      # log10(0) = -inf rows give NaN, as in the reference (Q5)
        out = ((times - sim_times[lo]) / span) * rows[:, hi] + ((sim_times[hi] - times) / span) * rows[:, lo]
    outside = (times < sim_times[0]) | (times > sim_times[-1])
    if outside.any():
        out[:, outside] = np.nan
    return out


def _thicknesses(sim_params, num_curves):
    if isinstance(sim_params[0], (list, tuple, np.ndarray)):
        return [float(v) for v in sim_params[0]]
    return [sim_params[0]] * num_curves


def _my_blocks(n, group, gpu_id, num_gpus):
    return [(b, min(group, n - b)) for b in range(gpu_id * group, n, num_gpus * group)]


def simulate(model, e_data, P, X, plI, plI_int, num_curves, sim_params, init_params, sim_flags,
             gpu_info, gpu_id, solver_time, err_sq_time, misc_time, logger=None):
    """Fill P[:, blocks of this gpu_id] (block-cyclic over gpu_info["num_gpus"] ranks in chunks of
    gpu_info["sims_per_gpu"], bayeslib.py:131)."""
    if not gpu_info.get("has_GPU", False):
        raise RuntimeError("the B200 engine needs a GPU (no CPU fallback)")
    if sim_flags["load_PL_from_file"]:
        raise NotImplementedError("load PL not implemented")
    dev = engine.require_cuda(gpu_info.get("device", None))
    group, num_gpus = gpu_info["sims_per_gpu"], gpu_info["num_gpus"]
    blocks = _my_blocks(len(X), group, gpu_id, num_gpus)
    thick = _thicknesses(sim_params, num_curves)
    log_pl, normalize = sim_flags["log_pl"], sim_flags["self_normalize"]
    if not blocks:
        return

    if gpu_info.get("fused", True):
        sp = list(sim_params)
        sp[0] = thick
        problem = engine.cached_problem(sp, init_params, e_data, device=dev.index)
        if len(blocks) == 1 or num_gpus == 1:
            lo, hi = blocks[0][0], blocks[-1][0] + blocks[-1][1]
            rows = slice(lo, hi)
            Xrows = X[lo:hi]
        else:
            rows = np.concatenate([np.arange(b, b + n) for b, n in blocks])
            Xrows = X[rows]
        # host -> pinned staging -> device, result device -> pinned -> P: one copy each way per call
        xh = engine.pinned("X", Xrows.shape, torch.float64)
        xh.numpy()[...] = Xrows
        clock0 = time.perf_counter()
        Xd = xh.to(dev, non_blocking=True)
        lnl, status, _ = engine.solve_loglik(Xd, problem, log_pl=log_pl, self_normalize=normalize,
                                             emulate_f32=gpu_info.get("emulate_f32", False))
        lh = engine.pinned("lnl", lnl.shape, torch.float64)
        sh = engine.pinned("status", status.shape, torch.int32)
        lh.copy_(lnl, non_blocking=True)
        sh.copy_(status, non_blocking=True)
        engine.host_wait(dev)
        solver_time[gpu_id] += time.perf_counter() - clock0
        P[:, rows] += lh.numpy()
        bad = int(np.count_nonzero(sh.numpy()))
        if bad and logger is not None:
            logger.warning("%d samples did not converge (lnL = NaN for them)", bad)
        return

    TPB = gpu_info["threads_per_block"]
    T = sim_params[3]
    sim_times = np.linspace(0, sim_params[1], T + 1)
    for ic_num in range(num_curves):
        sim_params[0] = thick[ic_num]
        for blk, size in blocks:
            if logger is not None:
                logger.info("Curve #%d: Calculating %d of %d", ic_num, blk, len(X))
            plI[gpu_id] = np.empty((size, T + 1), dtype=np.float32)
            solver_time[gpu_id] += model(plI[gpu_id], None, None, None, X[blk:blk + size, :-1],
                                         sim_params, init_params[ic_num], TPB, 0,
                                         gpu_info.get("max_sims_per_block", 1), init_mode="points")
            if normalize:
                plI[gpu_id] = (plI[gpu_id].T / plI[gpu_id].T[0]).T
            if log_pl:
                misc_time[gpu_id] += fastlog(plI[gpu_id], sys.float_info.min, TPB[0], 0)
            for e, exp in enumerate(e_data):
                times, values, std = exp[0][ic_num], exp[1][ic_num], exp[2][ic_num]
                if almost_equal(sim_times, times):
                    plI_int[gpu_id] = plI[gpu_id]
                else:
                    clock0 = time.perf_counter()
                    plI_int[gpu_id] = interpolate_rows(sim_times, plI[gpu_id], times)
                    misc_time[gpu_id] += time.perf_counter() - clock0
                err_sq_time[gpu_id] += prob(P[e, blk:blk + size], plI_int[gpu_id], values, std,
                                            np.ascontiguousarray(X[blk:blk + size, -1]), TPB[0], 0)


def rank_and_world():
    """(gpu_id, num_ranks) of this process: SLURM array task (the reference's launcher,
    bayeslib.py:231; the task count comes from SLURM_ARRAY_TASK_COUNT when SLURM exports it), else
    torchrun's RANK/WORLD_SIZE, else a single rank.  num_ranks is None when unknown."""
    if os.getenv("SLURM_ARRAY_TASK_ID") is not None:
        cnt = os.getenv("SLURM_ARRAY_TASK_COUNT")
        return int(os.getenv("SLURM_ARRAY_TASK_ID")), (int(cnt) if cnt is not None else None)
    if os.getenv("RANK") is not None:
        return int(os.getenv("RANK")), int(os.getenv("WORLD_SIZE", "1"))
    return 0, None


def override_flags(sim_flags):
    """Bit mask of the override_equal_* flags for the device samplers (1: mu, 2: s, 4: auger)."""
    return ((1 if sim_flags["override_equal_mu"] else 0) | (2 if sim_flags["override_equal_s"] else 0)
            | (4 if sim_flags["override_equal_auger"] else 0))


def _bayes_philox(N, num_exp, minX, maxX, do_log, init_params, sim_params, e_data, sim_flags, gpu_info, logger,
                  exchange=None):
    """sim_flags["sampler"] == "philox": every rank draws ONLY its own contiguous rows of the sample
    matrix on its GPU (counter-based Philox4x32-10, `first_sample` = first row of the shard, so the
    shards of any world size concatenate to the single-rank draw bit for bit), runs the fused path on
    them and the tables are all-gathered once at the end.  X never crosses PCIe on the way in; the
    bounds arrive already in engine units (parallel_bayes_gpu.py:183-184), so the unit conversion is
    part of the draw.  `exchange` (default: distributed.TorchExchange) supplies the rank and the gather."""
    from . import distributed
    ex = exchange if exchange is not None else distributed.TorchExchange()
    dev = engine.require_cuda(gpu_info.get("device", None))
    S = int(sim_flags["num_points"])
    rank, world = ex.rank_world()
    lo, hi = distributed.shard_bounds(S, rank, world)
    Xd = engine.random_grid_device(minX, maxX, do_log, hi - lo, int(sim_flags.get("seed", 42)),
                                   first_sample=lo, override_flags=override_flags(sim_flags), device=dev.index)
    problem = engine.cached_problem(list(sim_params), init_params, e_data, device=dev.index)
    lnl, status, _ = engine.solve_loglik(Xd, problem, log_pl=sim_flags["log_pl"],
                                         self_normalize=sim_flags["self_normalize"],
                                         emulate_f32=gpu_info.get("emulate_f32", False))
    bad = int((status != 0).sum().item())
    if bad and logger is not None:
        logger.warning("%d samples did not converge (lnL = NaN for them)", bad)
    P = ex.gather_rows(lnl, S)
    X = ex.gather_rows(Xd.t().contiguous(), S).t()
    return np.arange(S), P.cpu().numpy(), np.ascontiguousarray(X.cpu().numpy())


def bayes(model, N, P, minX, maxX, do_log, init_params, sim_params, e_data, sim_flags, gpu_info,
          logger=None, exchange=None):
    """Draw the sample matrix, evaluate this rank's share of the likelihood table, return
    (N, P, X) like bayeslib.bayes (bayeslib.py:207-252).  Columns of P that belong to other ranks
    stay 0 exactly as in the reference (bayes_io.py:134) -- except with sim_flags["sampler"] ==
    "philox", where the complete table comes back on every rank (gathered through `exchange`)."""
    if sim_flags.get("sampler", "numpy") == "philox":
        return _bayes_philox(N, len(e_data), minX, maxX, do_log, init_params, sim_params, e_data,
                             sim_flags, gpu_info, logger, exchange=exchange)
    num_gpus = gpu_info["num_gpus"]
    solver_time = np.zeros(num_gpus)
    err_sq_time = np.zeros(num_gpus)
    misc_time = np.zeros(num_gpus)
    num_curves = len(init_params)
    N, P, X = make_grid(N, P, len(e_data), minX, maxX, do_log, sim_flags)
    if logger is not None:
        logger.info("Initializing %d random samples", len(X))
    gpu_id, _ = rank_and_world()
    plI = [None] * num_gpus
    plI_int = [None] * num_gpus
    simulate(model, e_data, P, X, plI, plI_int, num_curves, list(sim_params), init_params,
             sim_flags, gpu_info, gpu_id, solver_time, err_sq_time, misc_time, logger=logger)
    if logger is not None:
        logger.info("Total tEvol time: %s, avg %s", solver_time, np.mean(solver_time))
        logger.info("Total err_sq time: %s, avg %s", err_sq_time, np.mean(err_sq_time))
        logger.info("Total misc time: %s, avg %s", misc_time, np.mean(misc_time))
    return N, P, X


def owned_columns(n, gpu_info, gpu_id):
    """Boolean mask of the columns of P this rank computed (block-cyclic layout, bayeslib.py:131)."""
    m = np.zeros(n, dtype=bool)
    for b, size in _my_blocks(n, gpu_info["sims_per_gpu"], gpu_id, gpu_info["num_gpus"]):
        m[b:b + size] = True
    return m
