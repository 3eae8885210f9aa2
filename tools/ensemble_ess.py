#!/usr/bin/env python3
"""Cost and statistical yield of the ensemble sampler on one GPU at the power-scan configuration (L=128,
T=80000 steps of 0.025 ns, Length 2000 nm, 3 power-scan curves, synthetic observations of the truth sample,
default prior with mobilities from 0.5): writes profiles/ensemble_ess.json.

  * per half-step, with CUDA events: the solve, and everything else (complement gather, proposals,
    accept/reject, chain bookkeeping, and the final gather + host copy of the chain, spread over the
    half-steps);
  * likelihoods/s of the ensemble path next to engine.solve_loglik on the same row count (W/2 prior draws);
  * effective samples per GPU-second: the ensemble's (integrated autocorrelation time per free parameter in
    prior coordinates, over the second half of the chain) and brute-force Philox sampling's
    ((sum w)^2 / sum w^2 with w = exp(lnL / temperature)) for the same number of likelihood evaluations.

    python tools/ensemble_ess.py [--walkers W] [--steps N] [--temperature T] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from bayesian_inference_trpl_b200 import engine, ensemble  # noqa: E402
from helpers import DO_LOG, MAXX, MINX, TRUTH, UC, power_scan_excitations  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return {"name": name, "power_limit": power}


def problem():
    L, T, Time, Length = 128, 80000, 2000.0, 2000.0
    inis = power_scan_excitations()
    m = torch.from_numpy((TRUTH * UC)[None, :12].copy()).cuda()
    grid = np.linspace(0, Time, T + 1)
    pls = [engine.solve_pl(m, torch.from_numpy(inis[c]).cuda(), Length, Time, L, T)[0][0].cpu().numpy()
           for c in range(3)]
    e_data = [([grid] * 3, [np.log10(p) for p in pls], [np.full(T + 1, 0.1)] * 3)]
    return engine.Problem([Length, Time, L, T, 1, (0,), 7, 10000], inis, e_data)


def integrated_time(x, c=5.0):
    """Integrated autocorrelation time of the walker-averaged autocorrelation function of x [steps, W]
    (Goodman & Weare 2010; automatic window M = smallest M >= c tau(M), Sokal)."""
    n = x.shape[0]
    f = np.fft.rfft(x - x.mean(axis=0), n=2 * n, axis=0)
    acf = np.fft.irfft(f * np.conj(f), axis=0)[:n].mean(axis=1)
    if not acf[0] > 0:
        return float("nan"), 0
    acf /= acf[0]
    taus = 2.0 * np.cumsum(acf) - 1.0
    m = np.arange(n) >= c * taus
    window = int(np.argmax(m)) if m.any() else n - 1
    return float(taus[window]), window


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--walkers", type=int, default=0, help="0: W/2 = two waves of resident simulations")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--temperature", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ensemble_ess.json"))
    args = ap.parse_args()
    info = card()
    prob = problem()
    resident = engine.resident_sims(128)
    W = args.walkers or 2 * (2 * resident // prob.C)
    W += W % 2
    lo, hi = MINX * UC, MAXX * UC
    lo[2:4] = 0.5 * UC[2]
    free = ensemble.free_columns(lo, hi)
    loglik = ensemble.solver_loglik(prob)
    steps, temp = args.steps, args.temperature

    # warm-up of every launch shape of the timed region
    X0 = ensemble.initial_walkers(W, lo, hi, DO_LOG, args.seed)
    ensemble.sample(X0, loglik, lo, hi, DO_LOG, 1, seed=args.seed + 1, temperature=temp)
    torch.cuda.synchronize()

    events = []

    def timer(tag):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        events.append((tag, ev))

    timer("start")
    chain = ensemble.sample(X0, loglik, lo, hi, DO_LOG, steps, seed=args.seed, temperature=temp, timer=timer)
    X, lnl, acc = chain.X.cpu().numpy(), chain.lnl.cpu().numpy(), chain.acceptance.cpu().numpy()
    timer("end")
    torch.cuda.synchronize()
    total = events[0][1].elapsed_time(events[-1][1]) * 1e-3
    solve = sum(a.elapsed_time(b) for (ta, a), (tb, b) in zip(events[1:-1], events[2:-1])
                if ta == "solve" and tb == "other") * 1e-3
    init_solve = events[1][1].elapsed_time(events[2][1]) * 1e-3       # all W walkers, once
    solve -= init_solve
    half_steps = 2 * steps
    other = total - solve - init_solve

    # engine.solve_loglik on the same row count (W/2 prior draws), and brute force with the same evaluations
    n_eval = W * (steps + 1)
    rows = W // 2
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    lnl_bf = []
    for b in range(0, n_eval, rows):
        Xb = engine.random_grid_device(lo, hi, DO_LOG, min(rows, n_eval - b), args.seed + 1000, first_sample=b)
        lnl_bf.append(loglik(Xb))
    t1.record()
    torch.cuda.synchronize()
    bf_time = t0.elapsed_time(t1) * 1e-3
    lbf = torch.cat(lnl_bf).cpu().numpy()
    ok = np.isfinite(lbf)
    w = np.exp((lbf[ok] - lbf[ok].max()) / temp)
    ess_bf = float(w.sum() ** 2 / (w ** 2).sum())

    post = X[steps // 2 + 1:]
    taus = {}
    for j in np.flatnonzero(free):
        col = np.log10(post[..., j]) if DO_LOG[j] else post[..., j]
        taus[int(j)] = integrated_time(col)
    tau_max = max(t for t, _ in taus.values())
    n_post = post.shape[0]
    ess_ens = W * n_post / tau_max
    res = {
        "card": info,
        "config": "power_scan L=128 T=80000 Length=2000nm 3 curves x 80001 obs, default prior (mobility >= 0.5), "
                  "synthetic observations of the truth sample",
        "walkers": W, "steps": steps, "temperature": temp, "free_parameters": int(free.sum()),
        "resident_sims": resident,
        "half_step_s": {"solve": solve / half_steps, "other": other / half_steps,
                        "other_fraction": other / (solve + other)},
        "initial_solve_s": init_solve,
        "ensemble_total_s": total,
        "likelihoods_per_s": {"ensemble_path": W * (steps + 1) / total,
                              "solve_loglik_same_rows_prior_draws": n_eval / bf_time},
        "acceptance": {"mean": float(acc.mean()), "last_half": float(acc[steps // 2:].mean()),
                       "per_step": [round(float(a), 4) for a in acc]},
        "median_lnL": {"step0": float(np.nanmedian(lnl[0])), "last": float(np.nanmedian(lnl[-1]))},
        "ensemble": {"tau_per_parameter": {str(j): {"tau": t, "window": m} for j, (t, m) in taus.items()},
                     "tau_max": tau_max, "post_burn_in_steps": n_post,
                     "tau_reliable": bool(n_post >= 50 * tau_max),
                     "ess": ess_ens, "ess_per_gpu_s": ess_ens / total},
        "brute_force": {"evaluations": n_eval, "time_s": bf_time, "ess": ess_bf, "ess_per_gpu_s": ess_bf / bf_time,
                        "nonfinite": int((~ok).sum())},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "acceptance"}, indent=1))


if __name__ == "__main__":
    main()
