#!/usr/bin/env python3
"""Benchmark of the fused forward-model + likelihood path: parameter-sample likelihoods per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--samples S]
                    [--impl ours|reference] [--no-cpu-baseline] [--no-reference-gpu] [--strong]
                    [--dump-outputs DIR]

Configurations (BASELINE.json `configs`, SURVEY.md 8(d)); `power_scan` is the headline and the default:
  power_scan  configs[1]: L=128, Length=2000 nm, T=80000 steps of 0.025 ns, 3 Power_scan excitations,
              default prior of the reference entry script, synthetic observations (PL of the truth
              sample, 80001 points per curve; the shipped file is missing from the reference mount)
  stiff       configs[2]: same grid, the 3 shipped stiff observation files in ONE call, prior widened to
              Sf,Sb in [1,1e5] cm/s; integration stops at each curve's last observation
  twothick    configs[3]: 6 curves, Length=[311,2000]x3, synthetic observations
  finegrid    configs[4]: L=1000, T=20000 (500 ns), 3 curves, synthetic observations (CTA-per-simulation kernel)

One "step" = one fused launch over S samples per GPU (default: 12 waves of resident simulations for the
128-node configurations, 4 waves of resident CTAs on the fine grid); the nominal 1M/4M/16M-sample
configurations are this step repeated.  Under torchrun every rank owns its own S samples (weak scaling, no data-path collective);
the only exchange -- all-gather of lnL + global log-sum-exp over NCCL -- happens ONCE, after the last
step, inside the timed region.  `strong` (N>1 or --strong) times one more step with a fixed global batch
of 8 x S samples split over the ranks.

`--dump-outputs DIR` writes what the last timed step returned to its caller: lnl.npy (the likelihood table
[E, S * ranks], float64), status.npy (per-sample solver status, float32) and, on more than one rank,
lse.npy (the global log-sum-exp of the first file's lnL, float64).  Inputs are seeded, so two
builds run with the same arguments can be compared output for output; the default batch S follows the
kernel's occupancy, so give --samples when the two builds may differ in occupancy.

`--impl reference` times the reference's own wired-in CPU path (bayeslib.simulate with has_GPU=False ->
pvSim_fallback.pvSim_cpu_fallback, SciPy BDF; parallel_bayes_gpu.py:157-163) from baseline/_ref, one
process per host core; the oracle port is used only if baseline/_ref is absent.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

TOL, MAXIT = 7, 10000
METRIC = "param-sample likelihoods/sec (3-curve power scan)"
UNIT = "likelihoods/s"
FLOP_STEP, FLOP_ITER = 29, 126          # per node: per time step / per Newton iteration (SURVEY App. B)
DUMP_BYTES = 60 * 2 ** 20               # cap of --dump-outputs: below 64 MB with the .npy headers
DUMP_NAMES = ("lnl", "status", "lse", "sample_index")


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def config_def(name):
    """Static description of a configuration: grid, curves, prior; observations are attached later
    (they need the engine for the synthetic ones)."""
    from helpers import example_data, power_scan_excitations
    if name == "power_scan":
        return dict(L=128, T=80000, Time=2000.0, lengths=[2000.0] * 3, inis=power_scan_excitations(),
                    stiff_prior=False, obs="synthetic",
                    desc="power_scan L=128 T=80000 Length=2000nm 3 curves x 80001 obs, default prior")
    if name == "stiff":
        return dict(L=128, T=80000, Time=2000.0, lengths=[2000.0] * 3, inis=power_scan_excitations(),
                    stiff_prior=True, obs="shipped",
                    desc="stiff L=128 dt=0.025ns 3 curves x 3 shipped observation files (Highfrontsurf/"
                         "Highbacksurf/Balancedhighsurf) in one call, prior Sf,Sb in [1,1e5] cm/s")
    if name == "twothick":
        ex = example_data()
        return dict(L=128, T=80000, Time=2000.0, lengths=[311.0, 2000.0] * 3, inis=ex["twothick_exc"] * 1e-21,
                    stiff_prior=False, obs="synthetic",
                    desc="twothick L=128 T=80000 6 curves Length=[311,2000]x3, 80001 obs per curve, default prior")
    if name == "finegrid":
        L = 1000
        xc = (np.arange(L) + 0.5) * (2000.0 / L)
        inis = np.stack([a * 1e-21 * np.exp(-6e-3 * xc) for a in (1.2738e16, 1.1539e17, 1.6485e18)])
        return dict(L=L, T=20000, Time=500.0, lengths=[2000.0] * 3, inis=inis, stiff_prior=False, obs="synthetic",
                    desc="finegrid L=1000 T=20000 (500 ns) Length=2000nm 3 curves x 20001 obs, default prior")
    raise SystemExit("unknown --config %s" % name)


def simpar_of(cfg, c=None):
    length = cfg["lengths"] if c is None else cfg["lengths"][c]
    if c is None and len(set(cfg["lengths"])) == 1:
        length = cfg["lengths"][0]
    return [length, cfg["Time"], cfg["L"], cfg["T"], 1, (0,), TOL, MAXIT]


def observations(cfg, trpl):
    """e_data for a configuration: shipped files, or PL of the truth sample from the engine itself."""
    from helpers import TRUTH, UC, example_data
    C = len(cfg["inis"])
    if cfg["obs"] == "shipped":
        ex = example_data()
        e_data = []
        for f in ("Highfrontsurf", "Highbacksurf", "Balancedhighsurf"):
            ts = [ex["%s_t%d" % (f, c)] for c in range(C)]
            vs = [np.log10(ex["%s_pl%d" % (f, c)] * 1e-23) for c in range(C)]
            e_data.append((ts, vs, [np.full(len(t), 0.1) for t in ts]))
        return e_data
    T, Time = cfg["T"], cfg["Time"]
    grid = np.linspace(0, Time, T + 1)
    ts, vs, us = [], [], []
    for c in range(C):
        pl = np.empty((1, T + 1))
        trpl.pvSim(pl, None, None, None, (TRUTH * UC)[None, :12], simpar_of(cfg, c), cfg["inis"][c], (128,), 0, 1,
                   init_mode="points")
        ts.append(grid.copy()); vs.append(np.log10(pl[0])); us.append(np.full(T + 1, 0.1))
    return [(ts, vs, us)]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows),
                "reasons": reasons}


def dump_outputs(out_dir, per_sample, whole=None):
    """Write host arrays as out_dir/<name>.npy: `per_sample` ones (last axis = parameter sample) and
    `whole` ones (small, written as they are).  Above DUMP_BYTES a fixed, seeded subset of samples is
    kept; its indices go to sample_index.npy.  Dump files of an earlier run that this run does not
    write are removed, so the directory always holds one run's outputs."""
    n = next(iter(per_sample.values())).shape[-1]
    per_row = sum(a.itemsize * (a.size // n) for a in per_sample.values())
    if per_row * n > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (per_row + 8), replace=False))
        per_sample = {name: a[..., keep] for name, a in per_sample.items()}
        per_sample["sample_index"] = keep.astype(np.float64)
    arrays = dict(per_sample, **(whole or {}))
    os.makedirs(out_dir, exist_ok=True)
    for name in DUMP_NAMES:
        if name not in arrays and os.path.exists(os.path.join(out_dir, name + ".npy")):
            os.remove(os.path.join(out_dir, name + ".npy"))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------------
# CPU baselines (rank 0, N=1): the oracle port and the reference's own CPU codes
# ------------------------------------------------------------------------------------------------
def port_rate(cfg, n_samples, threads, curves=None):
    """Oracle (C port of the reference algorithm, Thomas solve, OpenMP) -> (likelihoods/s, seconds)."""
    from helpers import prior_samples
    from oracle import oracle
    X = prior_samples(n_samples, seed=777, stiff=cfg["stiff_prior"])
    C = len(cfg["inis"])
    cs = range(C) if curves is None else curves
    t0 = time.perf_counter()
    for c in cs:
        oracle.solve(X[:, :12], simpar_of(cfg, c), cfg["inis"][c], solver="thomas", nthreads=threads)
    dt = time.perf_counter() - t0
    return n_samples * len(list(cs)) / C / dt, dt


def cpu_baselines(cfg, config_name, threads, with_reference=True):
    n_cpu = 4 * threads if cfg["L"] <= 128 else threads
    if config_name == "twothick":
        n_cpu = 2 * threads
    v, dt = port_rate(cfg, n_cpu, threads)
    C = len(cfg["inis"])
    out = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": "%d samples x %d curves at full T=%d (%.1f s), oracle/trpl_oracle.c Thomas solver, %d OpenMP threads"
                     % (n_cpu, C, cfg["T"], dt, threads)}
    if not (with_reference and config_name == "power_scan"):
        return out
    others = []
    try:
        from baseline import ref_runner as rr
        from helpers import prior_samples
        if not rr.available():
            raise RuntimeError("baseline/_ref not present")
        X = prior_samples(threads, seed=778)
        sp = simpar_of(cfg)
        # Legacy/pvSim.py: exponential-profile init (a, l) fitted to the three excitation rows
        amps = [(float(cfg["inis"][c][0]) * np.exp(6e-3 * 0.5 * 2000.0 / 128), 1.0 / 6e-3) for c in range(C)]
        lv, ldt = rr.legacy_njit_rate(X, sp, amps, threads)
        others.append({"impl": "Legacy/pvSim.py tEvol (numba njit; BDF2, no Auger: the reference's CPU twin of the GPU solver)",
                       "kind": "reference", "value": lv, "unit": UNIT, "cores": threads,
                       "sample": "%d samples x 3 curves at full T=80000 (%.1f s), one process per core" % (threads, ldt)})
        n_fb = max(16, threads)
        Xf = prior_samples(n_fb, seed=779, mag=False)
        fv, fdt = rr.fallback_rate(Xf, sp, cfg["inis"], threads)
        others.append({"impl": "pvSim_fallback.pvSim_cpu_fallback (SciPy BDF; the CPU model parallel_bayes_gpu.py wires in)",
                       "kind": "reference", "value": fv, "unit": UNIT, "cores": threads,
                       "sample": "%d samples x 3 curves, Time=2000 ns, T=80000 outputs (%.1f s), one process per core" % (n_fb, fdt)})
    except Exception as e:                                   # keep the bench line even if a reference leg fails
        others.append({"kind": "reference", "unavailable": repr(e)[:300]})
    out["others"] = others
    return out


def reference_gpu(cfg, S_ref=1024):
    """The reference's own numba-CUDA solver (baseline/_ref/pvSimPCR.py, unmodified) on this GPU."""
    try:
        from baseline import ref_runner as rr
        from helpers import prior_samples
        if not rr.available():
            return {"unavailable": "baseline/_ref not present on this box"}
        X = prior_samples(S_ref, seed=780)
        sp = simpar_of(cfg)
        rr.ref_pvsim(X[:8], [sp[0], 0.025 * 16, sp[2], 16, 1, (0,), TOL, MAXIT], cfg["inis"][0])     # JIT
        secs = []
        for c in range(len(cfg["inis"])):
            _, sec = rr.ref_pvsim(X, sp, cfg["inis"][c], dtype=np.float32)       # float32 PL buffer as bayeslib.py:137
            secs.append(sec)
        return {"value": S_ref / sum(secs), "unit": UNIT, "kind": "numba-cuda unmodified",
                "samples": S_ref, "curves": len(secs), "kernel_s": secs,
                "what": "pvSimPCR.pvSim tEvol kernel time only (BPG=8*SMs, TPB=128, one launch of %d samples per curve "
                        "= the reference's sims_per_gpu); its fastlog/interpolation/prob stages are NOT included" % S_ref}
    except Exception as e:
        return {"unavailable": repr(e)[:300]}


# ------------------------------------------------------------------------------------------------
# --impl reference: the reference's own CPU path
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = config_def(args.config)
    threads = host_threads()          # torchrun pins OMP_NUM_THREADS=1; use every core the process may run on
    C = len(cfg["inis"])
    from helpers import prior_samples
    use_ref = False
    try:
        from baseline import ref_runner as rr
        use_ref = rr.available() and args.config in ("power_scan", "stiff", "twothick")
    except Exception:
        use_ref = False
    times = []
    if use_ref:
        # one step = `threads` samples x ONE curve (a third of a likelihood each; the curve index rotates
        # with the step) so that a --steps 20 --warmup 5 run stays within minutes at ~7 s per curve
        import multiprocessing as mp
        X = prior_samples(threads, seed=777, stiff=cfg["stiff_prior"])
        chunks = [c for c in np.array_split(X, threads) if len(c)]
        with rr._one_thread_env(), mp.get_context("spawn").Pool(len(chunks)) as pool:
            def step(k):
                c = k % C
                t0 = time.perf_counter()
                pool.map(rr._fallback_worker, [(ch, simpar_of(cfg, c), [cfg["inis"][c]]) for ch in chunks])
                return time.perf_counter() - t0
            pool.map(rr._fallback_worker, [(ch[:0], simpar_of(cfg, 0), []) for ch in chunks])      # imports
            for k in range(min(args.warmup, 1)):
                step(k)
            for k in range(args.steps):
                times.append(step(k))
        n = threads / float(C)
        kind = "reference"
        sample = ("%d samples x 1 of %d curves per step (curve = step %% %d) at Time=%g ns / T=%d outputs, "
                  "pvSim_fallback.pvSim_cpu_fallback (SciPy BDF) from baseline/_ref, %d processes; "
                  "%d of the %d warm-up steps run (no GPU, nothing to warm beyond imports)"
                  % (threads, C, C, cfg["Time"], cfg["T"], threads, min(args.warmup, 1), args.warmup))
    else:
        n_s = max(threads, 1)
        for _ in range(min(args.warmup, 1)):
            port_rate(cfg, max(1, threads // 4), threads)
        for k in range(args.steps):
            _, dt = port_rate(cfg, n_s, threads)
            times.append(dt)
        n = n_s
        kind = "port"
        sample = "%d samples x %d curves at full T=%d per step, oracle Thomas solver, %d OpenMP threads" % (n_s, C, cfg["T"], threads)
    tot = sum(times)
    value = n * args.steps / tot
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": cfg["desc"], "config": args.config},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--samples", type=int, default=0, help="samples per GPU per step (0 = two waves of resident simulations)")
    ap.add_argument("--config", default="power_scan", choices=["power_scan", "stiff", "twothick", "finegrid"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--strong", action="store_true", help="also time one step of a fixed global batch (8 x S samples) split over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's lnL table and status as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference leg only times its CPU path")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import bayesian_inference_trpl_b200 as trpl
    from bayesian_inference_trpl_b200 import distributed as D
    from helpers import prior_samples

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = config_def(args.config)
    L, T, C = cfg["L"], cfg["T"], len(cfg["inis"])
    resident = trpl.engine.resident_sims(L, local)
    # default batch: 12 waves of resident simulations for the 128-node kernel (the tail of a launch, where
    # warps run out of work items, costs ~0.4 wave: 5 % at 6 waves, 2.5 % at 12, profiles/r02_variants.txt),
    # 4 waves of resident CTAs on fine grids
    S = args.samples if args.samples > 0 else max(1, 4 * resident * 3 // C) if L <= 256 else max(1, 4 * resident // C)
    X = prior_samples(S, seed=1234 + rank, stiff=cfg["stiff_prior"])
    e_data = observations(cfg, trpl)
    E = len(e_data)
    simPar = simpar_of(cfg)
    problem = trpl.engine.Problem(simPar, cfg["inis"], e_data, device=local)

    Xd = torch.from_numpy(X).pin_memory().to(dev)
    l2_flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    lnl_steps = torch.zeros((args.steps, E, S), dtype=torch.float64, device=dev)     # every step's table, exchanged once

    def exchange(tables):
        """The path's only exchange (SURVEY 8e): all-gather of per-sample lnL + global log-sum-exp.
        Returns (gathered tables, log-sum-exp of the last table's first file, or None on one rank)."""
        if world == 1:
            return tables, None
        flat = tables.reshape(-1, S)
        parts = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(parts, flat)
        lse = D.global_logsumexp(trpl.engine.lse_partial(tables[-1, 0].contiguous()))
        return torch.cat(parts, dim=-1), lse

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- warm-up (also yields the Newton totals for the flop count)
    for _ in range(max(args.warmup, 1)):
        l2_flush.zero_()
        lnl, status, iters = trpl.engine.solve_loglik(Xd, problem, want_iters=True)
    exchange(lnl_steps[:1])                      # NCCL communicator set-up and first-collective cost stay outside the timing
    torch.cuda.synchronize(dev)
    n_bad = int((status != 0).sum().item())
    iters_total = float(iters.sum().item())
    steps_per_sample = problem.steps_per_sample()
    flops_per_step = float(L * (FLOP_STEP * steps_per_sample * S + FLOP_ITER * iters_total))

    # ---- timed region: device-resident inputs, no per-step collective
    sampler = ClockSampler(local)
    sampler.start()
    kern_ev = []
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(args.steps):
        l2_flush.zero_()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        _, status_last, _ = trpl.engine.solve_loglik(Xd, problem, lnl=lnl_steps[k])
        k1.record()
        kern_ev.append((k0, k1))
    tables, lse = exchange(lnl_steps)
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    kern = [a.elapsed_time(b) for a, b in kern_ev]
    clocks = sampler.summary()

    # ---- end to end = the call a user of the reference makes: bayeslib.simulate(model, e_data, P, X, ...)
    # with HOST numpy arrays (bayeslib.py:83): stages X to the device, runs the fused kernel, reads lnL back
    # into P; the excitations / bracketed observations are staged on the first call with these arrays.
    sim_flags = {"load_PL_from_file": False, "log_pl": True, "self_normalize": False}
    gpu_info = {"has_GPU": True, "sims_per_gpu": S, "num_gpus": 1, "device": local,
                "threads_per_block": (128,), "max_sims_per_block": 1}
    P_host = np.zeros((E, S))
    obs_bytes = sum(len(t) * (4 + 8 + 8 + 8) for exp in e_data for t in exp[0])
    h2d_first = int(np.asarray(cfg["inis"]).size * 8 + obs_bytes)
    h2d_bytes = int(X.size * 8)
    d2h_bytes = int(E * S * 8 + S * 4)

    def step_e2e():
        P_host[:] = 0.0
        tm = [np.zeros(1), np.zeros(1), np.zeros(1)]
        trpl.bayeslib.simulate(trpl.pvSim, e_data, P_host, X, [None], [None], C, list(simPar), cfg["inis"],
                               sim_flags, gpu_info, 0, tm[0], tm[1], tm[2])
        return P_host

    step_e2e()                                   # warm the e2e path (problem staging, pinned buffers)
    e2e_steps = min(args.steps, 5)               # same per-step work as above; a handful of steps is enough
    p_tables = torch.zeros((e2e_steps, E, S), dtype=torch.float64, device=dev)
    p_stage = torch.zeros((e2e_steps, E, S), dtype=torch.float64).pin_memory()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(e2e_steps):
        l2_flush.zero_()
        step_e2e()
        p_stage[k].numpy()[...] = P_host         # the host-side tables of all steps, exchanged once at the end
    if world > 1:
        p_tables.copy_(p_stage, non_blocking=True)
        exchange(p_tables)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)

    # ---- strong scaling: fixed global batch of 8 x S samples, contiguous shards
    strong = None
    if args.strong or world > 1:
        G = 8 * S
        lo, hi = D.shard_bounds(G, rank, world)
        Xs = torch.from_numpy(prior_samples(G, seed=99, stiff=cfg["stiff_prior"])[lo:hi]).pin_memory().to(dev)
        tab = torch.zeros((1, E, hi - lo), dtype=torch.float64, device=dev)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        trpl.engine.solve_loglik(Xs, problem, lnl=tab[0])
        if world > 1:
            D.gather_rows(tab[0], G)
            D.global_logsumexp(trpl.engine.lse_partial(tab[0, 0].contiguous()))
        s1.record()
        barrier()
        strong = [s0.elapsed_time(s1), G]

    t = torch.tensor([ms_total, ms_e2e, float(np.mean(kern)), strong[0] if strong else 0.0],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, kern_mean, ms_strong = [float(v) for v in t.cpu()]

    if rank == 0:
        value = S * world * args.steps / (ms_total * 1e-3)
        e2e = S * world * e2e_steps / (ms_e2e * 1e-3)
        tf_peak, _ = trpl.engine.bench_dfma(20000, local)
        achieved = flops_per_step / (kern_mean * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        traffic, traffic_src = None, None
        if args.config == "power_scan":
            for name in ("r02_traffic.json", "r01_traffic.json"):
                try:   # DRAM bytes of one bench-sized launch, from a committed ncu --set full capture (not this run)
                    traffic = json.load(open(os.path.join(ROOT, "profiles", name)))["dram_bytes_per_launch"]
                    traffic_src = "committed ncu capture profiles/%s (a constant, not measured by this run)" % name
                    break
                except Exception:
                    pass
        kernel_name = "trpl_sim_kernel<%d,%s>" % (max(1, -(-L // 32)) if L <= 256 else 8, "pad" if L % 32 else "exact") \
            if L <= 256 else "trpl_sim_cta_kernel"
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["desc"], "config": args.config,
                       "batch": "%d samples/GPU/step out of the nominal configuration" % S,
                       "samples_per_gpu_per_step": S, "curves": C, "observation_files": E,
                       "time_steps_per_sample": steps_per_sample, "sims_resident_per_gpu": resident,
                       "l2": "256 MiB L2 flush between steps", "nonconverged_samples": n_bad,
                       "exchange": "one lnL all-gather + global log-sum-exp after the last step (inside the timed region)",
                       "mean_newton_iters_per_step": iters_total / (S * steps_per_sample)},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "h2d_bytes_first_call": h2d_first, "steps": e2e_steps,
                    "api": "bayeslib.simulate(model, e_data, P, X, ...) with host numpy arrays; excitations and "
                           "bracketed observations are staged once per (simPar, iniPar, e_data) and reused"},
            "gpu_launches": 2 * args.steps + (3 if world > 1 else 0),   # sim + finish per step (+ 3 lse kernels at the end when sharded)
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": achieved / tf_peak, "traffic": traffic, "traffic_source": traffic_src,
                         "note": "neither HBM- nor tensor-bound: scalar FP64 with no dense contraction "
                                 "(north_star); HBM side given in hbm_* keys, see DESIGN.md section 4",
                         "kernel": kernel_name, "kernel_ms": kern_mean, "flops_per_launch": flops_per_step,
                         "peak_source": "DFMA microbenchmark (trpl_bench_dfma) measured in this run; "
                                        "MEASURED_PEAKS.json has no FP64 entry",
                         "hbm_bytes_per_launch_algorithmic": int(S * (13 + E) * 8),
                         "hbm_peak_gbs_measured": peaks.get("hbm_gbs")},
        }
        if strong:
            out["strong"] = {"global_samples": strong[1], "ms": ms_strong, "value": strong[1] / (ms_strong * 1e-3),
                             "unit": UNIT, "note": "one step, fixed global batch split into contiguous shards, "
                                                   "lnL all-gather + log-sum-exp included"}
        if world == 1 and not args.no_reference_gpu and args.config == "power_scan":
            out["reference_gpu"] = reference_gpu(cfg)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baselines(cfg, args.config, host_threads())
        print(json.dumps(out))
    if args.dump_outputs:
        lnl_last = tables.reshape(-1, tables.shape[-1])[-E:]          # [E, S * world]: last step, all ranks
        if world > 1:
            parts = [torch.empty_like(status_last) for _ in range(world)]
            dist.all_gather(parts, status_last)
            status_last = torch.cat(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"lnl": lnl_last.cpu().numpy(),
                                             "status": status_last.cpu().numpy().astype(np.float32)},
                         {} if lse is None else {"lse": lse.cpu().numpy()})
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
