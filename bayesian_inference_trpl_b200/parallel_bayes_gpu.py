#!/usr/bin/env python3
"""Entry point mirroring the reference's `parallel_bayes_gpu.py` (config block :72-131, unit
conversion :27-33,183-194, bayes call :189, export :197-198) with the documented-but-never-
implemented command line (`README.md:4,29`: OBS EXC OUT) actually parsed.

    python -m bayesian_inference_trpl_b200.parallel_bayes_gpu EXC.csv OUT_DIR OBS.csv [OBS2.csv ...]
    torchrun --nproc-per-node 8 -m bayesian_inference_trpl_b200.parallel_bayes_gpu ...

Every rank draws the same sample matrix (global seed 42, parallel_bayes_gpu.py:35), evaluates
its block-cyclic share on its GPU with the fused kernel, the likelihood tables are merged over
NCCL and rank 0 writes <OUT>_BAYRAN_P.npy / _BAYRAN_X.npy (plus the normalised posterior
weights when --posterior is given).

With --sampler ensemble the posterior of ONE observation file is sampled by an ensemble MCMC instead
(stretch moves, ensemble.py): rank 0 writes the chain, <OUT>_MCMC_X.npy [steps+1, walkers, 13] in common
units and <OUT>_MCMC_P.npy [steps+1, walkers] (the untempered lnL).  With --ladder T0 T1 ... [inf] the
ensemble runs parallel tempering on that ladder (tempering.py): the two files hold the cold rung, and rank 0
also writes <OUT>_MCMC_PT_P.npy [steps+1, rungs, walkers] and <OUT>_MCMC_PT.json (per-rung mean lnL,
acceptance, swap acceptance, log-evidence)."""
import argparse
import json
import logging
import os
import sys
from time import perf_counter

import numpy as np

from . import bayes_io, bayes_validate, bayeslib, distributed
from .pvsim import pvSim

lambda0 = 704.3                           # q^2/(eps0*k_B T=25C) [nm]
param_names = ["n0", "p0", "mun", "mup", "B", "Sf", "Sb", "CN", "CP", "taun", "taup", "lambda",
               "mag_offset"]
# common units -> [V, nm, ns]
unit_conversions = np.array([(1e7) ** -3, (1e7) ** -3,
                             (1e7) ** 2 / (1e9) * .02569257, (1e7) ** 2 / (1e9) * .02569257,
                             (1e7) ** 3 / (1e9), (1e7) / (1e9), (1e7) / (1e9),
                             (1e7) ** 6 / (1e9), (1e7) ** 6 / (1e9), 1, 1, lambda0, 1])


def default_config():
    """The reference's hard-coded configuration (parallel_bayes_gpu.py:72-124)."""
    return {
        "Length": 311, "L": 2 ** 7, "Time": 2000, "T": 80000, "plT": 1, "pT": (0, 1, 3, 10, 30, 100),
        "tol": 7, "MAX": 10000,
        "do_log": np.array([1, 1, 0, 0, 1, 1, 1, 1, 1, 0, 0, 1, 0]),
        "minX": np.array([1e8, 1e14, 0, 0, 1e-11, 0.1, 0.1, 1e-30, 1e-30, 1, 1, 10 ** -1, 0]),
        "maxX": np.array([1e8, 1e16, 50, 50, 1e-9, 100, 100, 1e-28, 1e-28, 1000, 2000, 10 ** -1, 0]),
        "ic_flags": {"time_cutoff": 2000, "select_obs_sets": None, "noise_level": None},
        "gpu_info": {"sims_per_gpu": 2 ** 10, "num_gpus": 1},
        "sim_flags": {"load_PL_from_file": False, "override_equal_auger": False,
                      "override_equal_mu": False, "override_equal_s": False, "log_pl": True,
                      "self_normalize": False, "random_sample": True, "num_points": 2 ** 17,
                      "walkers": 1024, "steps": 100, "temperature": 1.0},
    }


def run(init_filename, experimental_data_filename, out_filename, cfg=None, seed=42, logger=None,
        posterior=False, exchange=None, nccl_id_file=None):
    """Same sequence as the reference `__main__` block; returns (P, X in common units).

    Launchers: (a) torchrun, one rank per GPU: the per-rank tables are merged over NCCL and rank 0
    exports; (b) SLURM array tasks like the reference (no communication): task k fills its
    block-cyclic columns and EVERY task exports, into `<out>_task<k>` when there is more than one
    task, with NaN in the columns it does not own (`merge_task_exports` joins them afterwards);
    the task count must agree with gpu_info["num_gpus"].

    `exchange` selects how the ranks of (a) exchange results: None or "torch" (torch.distributed, a
    process group over NCCL); "cabi" (an nccl.Communicator over the C ABI, no process group; a
    multi-rank run bootstraps it through the file `nccl_id_file`); or an object with the methods of
    distributed.TorchExchange, such as an open nccl.Communicator whose rank and size match
    RANK/WORLD_SIZE.  SLURM array tasks are not co-scheduled and always merge through files.

    cfg["sim_flags"]["sampler"] == "ensemble" samples the posterior of the one observation file with
    cfg["sim_flags"]["walkers"] walkers for ["steps"] steps at ["temperature"] (ensemble.sample) and returns
    (lnL chain [steps+1, W], X chain [steps+1, W, 13] in common units).  A ladder in
    cfg["sim_flags"]["ladder"] runs tempering.sample on it instead and returns the cold rung's chains."""
    import torch
    import torch.distributed as dist
    cfg = cfg or default_config()
    ensemble = cfg["sim_flags"].get("sampler", "numpy") == "ensemble"
    if ensemble and len(experimental_data_filename) != 1:
        raise ValueError("the ensemble sampler samples the posterior of one observation file; got %d (run one "
                         "ensemble per file)" % len(experimental_data_filename))
    if cfg["sim_flags"].get("ladder") is not None:
        if not ensemble:
            raise ValueError("a temperature ladder needs the ensemble sampler")
        if float(cfg["sim_flags"].get("temperature", 1.0)) != 1.0:
            raise ValueError("a temperature ladder and a sampling temperature exclude each other: the ladder's "
                             "first entry is the sampled temperature")
        from . import tempering
        tempering.check_ladder(cfg["sim_flags"]["ladder"])
    rank, world = bayeslib.rank_and_world()
    slurm = os.getenv("SLURM_ARRAY_TASK_ID") is not None
    if exchange == "cabi":
        with _cabi_communicator(rank, world, slurm, nccl_id_file) as comm:
            return run(init_filename, experimental_data_filename, out_filename, cfg=cfg, seed=seed, logger=logger,
                       posterior=posterior, exchange=comm)
    if exchange is None or exchange == "torch":
        if not slurm and world is not None and world > 1 and not dist.is_initialized():
            torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
            dist.init_process_group("nccl")
        exchange = distributed.TorchExchange()
    elif isinstance(exchange, str):
        raise ValueError("exchange must be 'torch', 'cabi' or an exchange object, not %r" % exchange)
    np.random.seed(seed)
    simPar = [cfg["Length"], cfg["Time"], cfg["L"], cfg["T"], cfg["plT"], cfg["pT"], cfg["tol"], cfg["MAX"]]
    ic_flags, sim_flags, gpu_info = cfg["ic_flags"], dict(cfg["sim_flags"]), dict(cfg["gpu_info"])
    sim_flags.setdefault("seed", seed)
    minX, maxX, do_log = cfg["minX"].astype(float).copy(), cfg["maxX"].astype(float).copy(), cfg["do_log"]

    iniPar = bayes_io.get_initpoints(init_filename, ic_flags)
    e_data = bayes_io.get_data(experimental_data_filename, ic_flags, sim_flags, logger=logger,
                               scale_f=1e-23)
    for exp in e_data:
        assert len(iniPar) == len(exp[0]), "Num. ICs mismatch num. datasets"
    bayes_validate.validate_ic_flags(ic_flags)
    bayes_validate.validate_IC(iniPar, cfg["L"])
    bayes_validate.validate_gpu_info(gpu_info)
    bayes_validate.validate_params(len(param_names), unit_conversions, do_log, minX, maxX)
    bayes_validate.connect_to_gpu(gpu_info, nthreads=128, sims_per_block=1)
    if not gpu_info["has_GPU"]:
        raise RuntimeError("no GPU: the B200 engine has no CPU fallback")
    if slurm:
        if world is not None and world != gpu_info["num_gpus"]:
            raise RuntimeError("SLURM_ARRAY_TASK_COUNT=%d disagrees with gpu_info['num_gpus']=%d: the tasks "
                               "would leave columns of P uncomputed" % (world, gpu_info["num_gpus"]))
        if rank >= gpu_info["num_gpus"]:
            raise RuntimeError("SLURM_ARRAY_TASK_ID=%d but gpu_info['num_gpus']=%d" % (rank, gpu_info["num_gpus"]))
        if sim_flags.get("sampler", "numpy") == "philox" and gpu_info["num_gpus"] > 1:
            raise RuntimeError("the philox sampler shards over torch.distributed ranks; use torchrun")
        if ensemble:
            raise RuntimeError("the ensemble sampler exchanges walkers every step, which SLURM array tasks "
                               "cannot do; use torchrun")
    elif world is not None:
        gpu_info["num_gpus"] = world

    minX *= unit_conversions
    maxX *= unit_conversions
    if ensemble:
        return _run_ensemble(iniPar, simPar, e_data, minX, maxX, do_log, sim_flags, gpu_info, out_filename[0],
                             exchange, logger)
    clock0 = perf_counter()
    N, P, X = bayeslib.bayes(pvSim, np.array([0]), None, minX, maxX, do_log, iniPar, simPar, e_data,
                             sim_flags, gpu_info, logger=logger, exchange=exchange)
    complete = sim_flags.get("sampler", "numpy") == "philox"
    if not complete and not slurm and world and world > 1:
        P = np.asarray(exchange.merge_block_cyclic(P).cpu())
    if logger is not None:
        logger.info("Bayesim took %.3f s", perf_counter() - clock0)
    X = X / unit_conversions
    outs = list(out_filename)
    if slurm and gpu_info["num_gpus"] > 1:
        mine = bayeslib.owned_columns(P.shape[1], gpu_info, rank)
        P = np.where(mine[None, :], P, np.nan)             # 0 would read as the best possible likelihood
        outs = ["%s_task%d" % (of.rstrip("/\\"), rank) for of in outs]
    if posterior:                                          # on every rank: the exchange may be collective
        W = [exchange.posterior_weights_full(torch.from_numpy(np.nan_to_num(P[i], nan=-np.inf)).cuda()).cpu().numpy()
             for i in range(len(outs))]
    if slurm or rank == 0:
        for i, of in enumerate(outs):
            bayes_io.export(of, P[i], X, logger=logger)
            if posterior:
                np.save(os.path.join(of, os.path.basename(os.path.normpath(of)) + "_BAYRAN_W.npy"), W[i])
    return P, X


def _run_ensemble(iniPar, simPar, e_data, minX, maxX, do_log, sim_flags, gpu_info, out, exchange, logger):
    """run() with sampler "ensemble": bounds in engine units; rank 0 writes <out>_MCMC_[XP].npy."""
    from . import engine, ensemble
    rank, world = exchange.rank_world()
    dev = engine.require_cuda(gpu_info.get("device", None))
    W, steps, seed = int(sim_flags["walkers"]), int(sim_flags["steps"]), int(sim_flags["seed"])
    flags = bayeslib.override_flags(sim_flags)
    problem = engine.cached_problem(list(simPar), iniPar, e_data, device=dev.index)
    loglik = ensemble.solver_loglik(problem, log_pl=sim_flags["log_pl"], self_normalize=sim_flags["self_normalize"],
                                    emulate_f32=gpu_info.get("emulate_f32", False))
    if sim_flags.get("ladder") is not None:
        return _run_tempered(loglik, minX, maxX, do_log, W, steps, seed, flags, sim_flags["ladder"], dev, out,
                             exchange, logger)
    X0 = ensemble.initial_walkers(W, minX, maxX, do_log, seed, flags, rank, world, device=dev.index)
    clock0 = perf_counter()
    chain = ensemble.sample(X0, loglik, minX, maxX, do_log, steps, n_walkers=W, override_flags=flags,
                            temperature=float(sim_flags["temperature"]), seed=seed, exchange=exchange)
    P, X = chain.lnl.cpu().numpy(), chain.X.cpu().numpy() / unit_conversions
    acc = chain.acceptance.cpu().numpy()
    if logger is not None:
        logger.info("ensemble: %d walkers x %d steps on %d rank(s) took %.3f s; acceptance fraction %.3f overall, "
                    "%.3f over the last half", W, steps, world, perf_counter() - clock0,
                    acc.mean() if steps else float("nan"), acc[steps // 2:].mean() if steps else float("nan"))
    if rank == 0:
        os.makedirs(out, exist_ok=True)
        base = os.path.basename(os.path.normpath(out))
        np.save(os.path.join(out, base + "_MCMC_X.npy"), X)
        np.save(os.path.join(out, base + "_MCMC_P.npy"), P)
        if logger is not None:
            logger.info("wrote %s_MCMC_[XP].npy to %s", base, out)
    return P, X


def _run_tempered(loglik, minX, maxX, do_log, W, steps, seed, flags, ladder, dev, out, exchange, logger):
    """_run_ensemble on a temperature ladder: rank 0 writes the cold rung to <out>_MCMC_[XP].npy, every rung's
    lnL to <out>_MCMC_PT_P.npy and the summary (log-evidence over the second half) to <out>_MCMC_PT.json."""
    from . import tempering
    rank, world = exchange.rank_world()
    T = tempering.check_ladder(ladder)
    K = T.shape[0]
    X0 = tempering.initial_walkers(W, K, minX, maxX, do_log, seed, flags, rank, world, device=dev.index)
    clock0 = perf_counter()
    chain = tempering.sample(X0, loglik, minX, maxX, do_log, steps, T, n_walkers=W, override_flags=flags, seed=seed,
                             exchange=exchange)
    PT, X = chain.lnl.cpu().numpy(), chain.X.cpu().numpy() / unit_conversions
    acc, swp = chain.acceptance.cpu().numpy(), chain.swap_acceptance.cpu().numpy()
    burn = steps // 2
    ev = tempering.log_evidence(PT, T, burn)
    if logger is not None:
        logger.info("tempered ensemble: %d rungs x %d walkers x %d steps on %d rank(s) took %.3f s; ln Z = %.6g "
                    "+- %.3g", K, W, steps, world, perf_counter() - clock0, ev.lnZ, ev.err)
    if rank == 0:
        os.makedirs(out, exist_ok=True)
        base = os.path.join(out, os.path.basename(os.path.normpath(out)))
        np.save(base + "_MCMC_X.npy", X)
        np.save(base + "_MCMC_P.npy", PT[:, 0])
        np.save(base + "_MCMC_PT_P.npy", PT)

        def num(v):
            return [num(u) for u in v] if np.ndim(v) else (float(v) if np.isfinite(v) else str(float(v)))
        summary = {"temperatures": num(T), "walkers": W, "steps": steps, "burn": burn,
                   "mean_lnl": num(ev.mean_lnl),
                   "acceptance": num(acc[burn:].mean(axis=0) if steps else np.full(K, np.nan)),
                   "swap_acceptance": num(swp[burn:].mean(axis=0) if steps else np.full(K - 1, np.nan)),
                   "log_evidence": num(ev.lnZ), "log_evidence_err": num(ev.err),
                   "beta_min_extrapolated": ev.extrapolated, "prior_rung": bool(np.isinf(T[-1])),
                   "nonfinite_lnl": int((~np.isfinite(PT)).sum())}
        with open(base + "_MCMC_PT.json", "w") as fh:
            json.dump(summary, fh, indent=1)
        if logger is not None:
            logger.info("wrote %s_MCMC_[XP].npy, _MCMC_PT_P.npy and _MCMC_PT.json to %s", os.path.basename(base),
                        out)
    return PT[:, 0], X


def _cabi_communicator(rank, world, slurm, nccl_id_file):
    """nccl.Communicator of this rank for run(..., exchange="cabi"): rank and size from RANK/WORLD_SIZE, the
    GPU from LOCAL_RANK, like torchrun; a single process needs no id file."""
    import torch
    from . import nccl
    if slurm:
        raise RuntimeError("SLURM array tasks are not co-scheduled, so NCCL cannot join them: they merge "
                           "through files (merge_task_exports)")
    if world is None or world == 1:
        return nccl.Communicator(nccl.unique_id(), 0, 1, torch.cuda.current_device())
    if not nccl_id_file:
        raise ValueError("exchange='cabi' with %d ranks needs an id file every rank can read (--nccl-id-file)"
                         % world)
    device = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(device)
    return nccl.Communicator.from_file(nccl_id_file, rank, world, device)


def merge_task_exports(out_filename, num_tasks):
    """Join the `<out>_task<k>` exports of a SLURM array run into `<out>`: every column is taken from
    the task that owns it (the others hold NaN there); a column nobody computed stays NaN."""
    base = os.path.basename(os.path.normpath(out_filename))
    P, X = None, None
    for k in range(num_tasks):
        d = "%s_task%d" % (out_filename.rstrip("/\\"), k)
        b = os.path.basename(os.path.normpath(d))
        Pk = np.load(os.path.join(d, b + "_BAYRAN_P.npy"))
        X = np.load(os.path.join(d, b + "_BAYRAN_X.npy"))
        P = Pk.copy() if P is None else np.where(np.isnan(P), Pk, P)
    bayes_io.export(out_filename, P, X)
    return P, X


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("excitations")
    ap.add_argument("out")
    ap.add_argument("observations", nargs="+")
    ap.add_argument("--num-points", type=int, default=None)
    ap.add_argument("--length", type=float, nargs="+", default=None, help="film thickness(es) in nm")
    ap.add_argument("--time-steps", type=int, default=None)
    ap.add_argument("--final-time", type=float, default=None)
    ap.add_argument("--posterior", action="store_true", help="also write normalised posterior weights")
    ap.add_argument("--sampler", choices=["numpy", "philox", "ensemble"], default="numpy",
                    help="numpy: the reference's host draw (np.random.seed(42), bit-compatible); philox: every rank "
                         "draws only its own rows on its GPU; ensemble: MCMC with stretch moves (one observation "
                         "file), writes the chain to <out>_MCMC_X.npy / _MCMC_P.npy")
    ap.add_argument("--walkers", type=int, default=None, help="ensemble: number of walkers (even)")
    ap.add_argument("--steps", type=int, default=None, help="ensemble: number of steps")
    ap.add_argument("--temperature", type=float, default=None,
                    help="ensemble: sample exp(lnL / temperature) (default 1)")
    ap.add_argument("--ladder", type=float, nargs="+", default=None, metavar="T",
                    help="ensemble: parallel tempering on these temperatures (strictly increasing from T0 > 0, the "
                         "last may be inf = the prior); writes the cold rung as without it, plus "
                         "<out>_MCMC_PT_P.npy and <out>_MCMC_PT.json with the log-evidence")
    ap.add_argument("--sims-per-gpu", type=int, default=None)
    ap.add_argument("--exchange", choices=["torch", "cabi"], default="torch",
                    help="how torchrun ranks exchange results: torch.distributed, or the NCCL C ABI "
                         "(libtrpl_b200_nccl.so) without a process group")
    ap.add_argument("--nccl-id-file", default=None,
                    help="with --exchange cabi and several ranks: a path every rank can read, which must not "
                         "exist yet; rank 0 writes the communicator id there")
    args = ap.parse_args(argv)
    logging.basicConfig(level=logging.INFO, format="%(asctime)s %(levelname)s: %(message)s")
    logger = logging.getLogger("Bayes Logger Main")
    cfg = default_config()
    if args.num_points:
        cfg["sim_flags"]["num_points"] = args.num_points
    cfg["sim_flags"]["sampler"] = args.sampler
    for key in ("walkers", "steps", "temperature"):
        if getattr(args, key) is not None:
            cfg["sim_flags"][key] = getattr(args, key)
    if args.ladder is not None:
        from . import tempering
        if args.sampler != "ensemble":
            ap.error("--ladder needs --sampler ensemble")
        if args.temperature is not None:
            ap.error("--ladder and --temperature exclude each other: the ladder's first entry is the sampled "
                     "temperature")
        try:
            cfg["sim_flags"]["ladder"] = list(tempering.check_ladder(args.ladder))
        except ValueError as e:
            ap.error("--ladder: %s" % e)
    if args.sims_per_gpu:
        cfg["gpu_info"]["sims_per_gpu"] = args.sims_per_gpu
    if args.length:
        cfg["Length"] = args.length[0] if len(args.length) == 1 else list(args.length)
    if args.time_steps:
        cfg["T"] = args.time_steps
    if args.final_time:
        cfg["Time"] = args.final_time
        cfg["ic_flags"]["time_cutoff"] = args.final_time
    outs = [args.out] if len(args.observations) == 1 else \
        [args.out + "_%d" % i for i in range(len(args.observations))]
    run(args.excitations, args.observations, outs, cfg=cfg, logger=logger, posterior=args.posterior,
        exchange=args.exchange, nccl_id_file=args.nccl_id_file)


if __name__ == "__main__":
    main(sys.argv[1:])
