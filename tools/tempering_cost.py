#!/usr/bin/env python3
"""Cost and yield of parallel tempering on one GPU at the power-scan configuration (the problem and prior of
tools/ensemble_ess.py): writes profiles/tempering.json.

Two runs in the same process, after a warm-up of every launch shape, with the same rows per solve and so the
same number of likelihood evaluations:
  * tempering.sample with K rungs of W walkers (default 8 x 400: K W / 2 = 1 600 rows, about two resident
    waves per half-step) on a geometric ladder from 1 to t_max over K - 1 rungs plus T = inf;
  * ensemble.sample with K W walkers.
Reported: per half-step, with CUDA events, the solve and everything else (gather, propose, accept, swap,
chain bookkeeping, final gather and host copy spread over the half-steps); likelihoods/s of both runs; the
acceptance per rung and swap acceptance per pair; the cold rung's median and maximum lnL per step beside the
plain run's; ln Z +- err (second half of the chain).

    python tools/tempering_cost.py [--rungs K] [--walkers W] [--t-max T] [--steps N] [--out PATH]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bayesian_inference_trpl_b200 import ensemble, tempering  # noqa: E402
from ensemble_ess import card, problem  # noqa: E402
from helpers import DO_LOG, MAXX, MINX, UC  # noqa: E402


def timed(run):
    """run(timer) under CUDA events: (result, total s, solve s excluding the initial solve, initial solve s)."""
    events = []

    def timer(tag):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        events.append((tag, ev))

    timer("start")
    res = run(timer)
    res = [r.cpu().numpy() if isinstance(r, torch.Tensor) else r for r in res]
    timer("end")
    torch.cuda.synchronize()
    total = events[0][1].elapsed_time(events[-1][1]) * 1e-3
    solve = sum(a.elapsed_time(b) for (ta, a), (tb, b) in zip(events[1:-1], events[2:-1])
                if ta == "solve" and tb == "other") * 1e-3
    init = events[1][1].elapsed_time(events[2][1]) * 1e-3
    return res, total, solve - init, init


def per_step(lnl):
    with np.errstate(all="ignore"):
        return {"median": [round(float(v), 3) for v in np.nanmedian(lnl, axis=1)],
                "max": [round(float(v), 3) for v in np.nanmax(lnl, axis=1)]}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rungs", type=int, default=8)
    ap.add_argument("--walkers", type=int, default=400, help="walkers per rung")
    ap.add_argument("--t-max", type=float, default=5e4, help="hottest finite temperature")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tempering.json"))
    args = ap.parse_args()
    info = card()
    prob = problem()
    lo, hi = MINX * UC, MAXX * UC
    lo[2:4] = 0.5 * UC[2]
    loglik = ensemble.solver_loglik(prob)
    K, W, steps, seed = args.rungs, args.walkers, args.steps, args.seed
    T = tempering.geometric_ladder(K, args.t_max)
    Xpt = tempering.initial_walkers(W, K, lo, hi, DO_LOG, seed)
    Xens = ensemble.initial_walkers(K * W, lo, hi, DO_LOG, seed)

    def run_pt(n, timer=None, s=seed):
        return tempering.sample(Xpt, loglik, lo, hi, DO_LOG, n, T, seed=s, timer=timer)

    def run_ens(n, timer=None, s=seed):
        return ensemble.sample(Xens, loglik, lo, hi, DO_LOG, n, seed=s, timer=timer)

    run_pt(1, s=seed + 1)                               # warm-up of every launch shape of the timed regions
    run_ens(1, s=seed + 1)
    torch.cuda.synchronize()
    print("warm-up done; %d steps of %d rungs x %d walkers" % (steps, K, W), flush=True)
    (_, pt_lnl, pt_acc, pt_swap, _), pt_total, pt_solve, pt_init = timed(lambda tm: run_pt(steps, tm))
    print("tempered: %.1f s; plain ensemble of %d walkers next" % (pt_total, K * W), flush=True)
    (_, ens_lnl, ens_acc), ens_total, ens_solve, ens_init = timed(lambda tm: run_ens(steps, tm))
    burn = steps // 2
    ev = tempering.log_evidence(pt_lnl, T, burn)
    half_steps = 2 * steps

    def cost(total, solve, init, evaluations):
        other = total - solve - init
        return {"half_step_s": {"solve": solve / half_steps, "other": other / half_steps,
                                "other_fraction": other / (solve + other)},
                "initial_solve_s": init, "total_s": total, "likelihoods_per_s": evaluations / total}

    res = {
        "card": info,
        "config": "power_scan L=128 T=80000 Length=2000nm 3 curves x 80001 obs, default prior (mobility >= 0.5), "
                  "synthetic observations of the truth sample",
        "steps": steps, "burn": burn, "seed": seed, "rows_per_solve": K * W // 2,
        "tempered": dict(cost(pt_total, pt_solve, pt_init, K * W * (steps + 1)), rungs=K, walkers_per_rung=W,
                         temperatures=[float(t) if np.isfinite(t) else "inf" for t in T],
                         acceptance_per_rung=[round(float(a), 4) for a in pt_acc[burn:].mean(axis=0)],
                         swap_acceptance_per_pair=[round(float(a), 4) for a in pt_swap[burn:].mean(axis=0)],
                         swap_acceptance_per_pair_all_steps=[round(float(a), 4) for a in pt_swap.mean(axis=0)],
                         mean_lnl_per_rung=[float(m) for m in ev.mean_lnl],
                         log_evidence=ev.lnZ, log_evidence_err=ev.err, nonfinite_lnl=int((~np.isfinite(pt_lnl)).sum()),
                         cold_lnl_per_step=per_step(pt_lnl[:, 0])),
        "plain": dict(cost(ens_total, ens_solve, ens_init, K * W * (steps + 1)), walkers=K * W,
                      acceptance=round(float(ens_acc[burn:].mean()), 4), lnl_per_step=per_step(ens_lnl)),
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    summary = {k: v for k, v in res.items() if k not in ("tempered", "plain")}
    for k in ("tempered", "plain"):
        summary[k] = {a: b for a, b in res[k].items() if not a.endswith("per_step")}
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
