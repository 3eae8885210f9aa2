"""Parallel tempering of the ensemble sampler (tempering.py, include/trpl_b200_tempering.h): the binding agrees
with the header, bad ladders and arguments are refused before the device is entered, the ladder and
log-evidence host rules hold, and the command line refuses bad options; on a GPU the three kernels agree with
host mirrors, one rung reduces to the untempered sampler bit for bit, the chain does not depend on the number
of ranks, every rung samples its tempered target, a two-mode target gets its mode weights right where the
untempered sampler does not, and the command line writes the tempered chain."""
import ctypes
import json
import os
import re
import threading

import numpy as np
import pytest

from helpers import DO_LOG
from test_ensemble import (MASK, _cli_args, _engine_prior, _header, _mcmc, _prior_rows, _small_problem,
                           _ThreadExchange, mirror_log_u, mirror_propose, philox)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "trpl_b200_tempering.h")

EINVAL, ENODEVICE = -1, -4
P = ctypes.c_void_p(16)          # placeholder device pointer: no case below dereferences it
INF, NAN = float("inf"), float("nan")


@pytest.fixture(scope="module")
def tlib():
    import bayesian_inference_trpl_b200 as trpl
    trpl.build()
    return trpl.tempering.lib()


def test_binding_matches_header(tlib, monkeypatch):
    import test_ensemble
    from bayesian_inference_trpl_b200 import _lib, ensemble, tempering
    monkeypatch.setattr(test_ensemble, "HEADER", HEADER)
    funcs = _header()
    assert list(funcs) == tempering.EXPORTS == ["trpl_tempered_propose", "trpl_tempered_accept",
                                                "trpl_tempered_swap"]
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name, (ret, params) in funcs.items():
        assert hasattr(raw, name), name
        restype, argtypes = tempering._SIGNATURES[name]
        assert restype is test_ensemble._ctype(ret), name
        assert [test_ensemble._ctype(p) for p in params] == argtypes, name
        fn = getattr(tlib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name
    assert set(_lib.EXPORTS).isdisjoint(funcs) and set(ensemble.EXPORTS).isdisjoint(funcs)
    defines = dict(re.findall(r"#define\s+(TRPL_\w+)\s+(\d+)", open(HEADER).read()))
    assert int(defines["TRPL_MAX_RUNGS"]) == tempering.MAX_RUNGS
    assert int(defines["TRPL_TAG_SWAP"]) == tempering.TAG_SWAP


def _ladder(temps):
    T = np.asarray(temps, dtype=np.float64)
    return T, (T.ctypes.data if T.size else None)


def _propose(lib, K=2, d_x=P, n=4, W=32, first=0, device=-1):
    lo, hi = np.zeros(17), np.ones(17)
    lo[0] = hi[0] = 0.5
    dl = np.zeros(17, dtype=np.int32)
    return lib.trpl_tempered_propose(d_x, n, 17, first, W, K, P, 64, lo.ctypes.data, hi.ctypes.data, dl.ctypes.data,
                                     13, 0, 2.0, 1, 0, P, 17, P, device, None)


def _accept(lib, temps=(1.0, 2.0), K=None, d_lnl=P, n=4, W=32, first=0, device=-1):
    T, ptr = _ladder(temps)
    return lib.trpl_tempered_accept(P, n, 17, first, W, len(temps) if K is None else K, ptr, 13, d_lnl, P, 17, P, P,
                                    1, 0, None, device, None)


def _swap(lib, temps=(1.0, 2.0), K=None, d_x=P, n=4, W=32, first=0, ncol=13, device=-1):
    T, ptr = _ladder(temps)
    return lib.trpl_tempered_swap(d_x, n, 17, first, W, len(temps) if K is None else K, ptr, ncol, P, 1, 0, None,
                                  device, None)


BAD_LADDERS = [(2.0, 1.0), (1.0, 1.0), (0.0, 1.0), (-1.0, 2.0), (1.0, NAN), (NAN, 2.0), (1.0, INF, 5.0),
               (INF, INF), ()]


def test_return_code_contract(tlib):
    cases = [
        (_propose(tlib, K=0), EINVAL),
        (_propose(tlib, K=65), EINVAL),
        (_propose(tlib, d_x=None), EINVAL),
        (_propose(tlib, W=22), EINVAL),                 # fewer than 2 x 12 free columns
        (_propose(tlib, first=14), EINVAL),             # crosses from half A into half B
        (_propose(tlib), ENODEVICE),
        (_propose(tlib, K=64), ENODEVICE),
        (_accept(tlib, d_lnl=None), EINVAL),
        (_accept(tlib, temps=(1.0,), K=0), EINVAL),
        (_accept(tlib, temps=tuple(range(1, 66))), EINVAL),
        (_accept(tlib, first=29), EINVAL),
        (_accept(tlib), ENODEVICE),
        (_accept(tlib, temps=(1.0, 3.0, INF)), ENODEVICE),
        (_accept(tlib, temps=(INF,)), ENODEVICE),
        (_accept(tlib, temps=tuple(range(1, 65))), ENODEVICE),
        (_swap(tlib, d_x=None), EINVAL),
        (_swap(tlib, ncol=17), EINVAL),
        (_swap(tlib, temps=(1.0,), K=0), EINVAL),
        (_swap(tlib, W=31), EINVAL),
        (_swap(tlib), ENODEVICE),
        (_swap(tlib, temps=(0.5, 1.0, 8.0, INF)), ENODEVICE),
        (_swap(tlib, temps=tuple(range(1, 66))), EINVAL),
        (_swap(tlib, temps=tuple(range(1, 65))), ENODEVICE),
    ]
    cases += [(_accept(tlib, temps=t), EINVAL) for t in BAD_LADDERS]
    cases += [(_swap(tlib, temps=t), EINVAL) for t in BAD_LADDERS]
    assert [rc for rc, _ in cases] == [want for _, want in cases]


def test_propose_refuses_a_complement_without_every_rung():
    import torch
    from bayesian_inference_trpl_b200 import tempering
    lo, hi = np.zeros(13), np.ones(13)
    X = torch.zeros((2 * 4, 13), dtype=torch.float64)   # K = 2 rungs of 4 walkers, never reaches the device
    for comp in (torch.zeros((13, 16), dtype=torch.float64), torch.zeros((26, 15), dtype=torch.float64)):
        with pytest.raises(ValueError, match="every rung's complement"):
            tempering.propose(X, 0, 32, 2, comp, lo, hi, np.zeros(13, dtype=np.int32))


def test_check_and_geometric_ladder():
    from bayesian_inference_trpl_b200 import tempering
    for bad in BAD_LADDERS + [tuple(range(1, 66))]:
        with pytest.raises(ValueError):
            tempering.check_ladder(bad)
    assert list(tempering.check_ladder([1, 2.5, INF])) == [1.0, 2.5, INF]
    np.testing.assert_allclose(tempering.geometric_ladder(5, 1000.0, prior_rung=False),
                               [1.0, 10 ** 0.75, 10 ** 1.5, 10 ** 2.25, 1000.0], rtol=1e-14)
    T = tempering.geometric_ladder(8, 5e4)
    assert T.shape == (8,) and T[0] == 1.0 and T[6] == 5e4 and T[7] == INF
    np.testing.assert_allclose(T[1:7] / T[:6], 5e4 ** (1 / 6), rtol=1e-13)
    assert list(tempering.geometric_ladder(2, 123.0)) == [1.0, INF]
    assert list(tempering.geometric_ladder(1, 123.0, prior_rung=False)) == [1.0]
    for args in ((1, 10.0), (0, 10.0, False), (3, 1.0, False)):
        with pytest.raises(ValueError):
            tempering.geometric_ladder(*args)


def test_log_evidence_rules():
    from bayesian_inference_trpl_b200 import tempering
    T = np.array([1.0, 2.0, 4.0, 8.0, INF])
    means = np.array([-1.0, -3.0, -6.0, -20.0, -100.0])
    lnl = np.broadcast_to(means[None, :, None], (6, 5, 4)).copy()
    lnl[:3] = 7.0                                       # before burn: ignored
    lnl[3, 2, 0], lnl[4, 2, 1], lnl[5, 0, 3] = NAN, -INF, INF     # non-finite entries are skipped
    ev = tempering.log_evidence(lnl, T, burn=3)
    np.testing.assert_array_equal(ev.mean_lnl, means)
    b = [1.0, 0.5, 0.25, 0.125, 0.0]
    want = sum((b[t] - b[t + 1]) * (means[t] + means[t + 1]) / 2 for t in range(4))
    assert ev.lnZ == pytest.approx(want, rel=1e-15) and not ev.extrapolated
    coarse = (1.0 - 0.25) * (-1.0 - 6.0) / 2 + 0.25 * (-6.0 - 100.0) / 2          # rungs 0, 2, 4
    assert ev.err == pytest.approx(abs(want - coarse), rel=1e-14)
    # a finite hottest rung: the segment [0, beta_min] is beta_min x its mean; rungs 0, 2, 3 keep both ends
    ev = tempering.log_evidence(lnl[:, :4], T[:4], burn=3)
    want = sum((b[t] - b[t + 1]) * (means[t] + means[t + 1]) / 2 for t in range(3)) + 0.125 * -20.0
    coarse = 0.75 * (-7.0) / 2 + 0.125 * (-26.0) / 2 + 0.125 * -20.0
    assert ev.extrapolated and ev.lnZ == pytest.approx(want, rel=1e-15)
    assert ev.err == pytest.approx(abs(want - coarse), rel=1e-14)
    # one rung at T_0 = 1: ln Z = <lnL>, no error estimate; a rung without finite entries gives NaN
    ev = tempering.log_evidence(lnl[:, :1], T[:1], burn=3)
    assert ev.lnZ == -1.0 and ev.err == 0.0 and ev.extrapolated
    lnl[:, 1] = NAN
    assert np.isnan(tempering.log_evidence(lnl, T, burn=3).lnZ)
    with pytest.raises(ValueError):
        tempering.log_evidence(lnl, T[:3], burn=0)


@pytest.mark.parametrize("extra, message", [
    (["--sampler", "numpy", "--ladder", "1", "10"], "needs --sampler ensemble"),
    (["--sampler", "ensemble", "--ladder", "1", "10", "--temperature", "2"], "exclude each other"),
    (["--sampler", "ensemble", "--ladder", "1", "10", "5"], "strictly increasing"),
    (["--sampler", "ensemble", "--ladder", "1", "inf", "10"], "strictly increasing"),
    (["--sampler", "ensemble", "--ladder", "0", "10"], "strictly increasing"),
])
def test_cli_rejects_bad_ladder_options(tmp_path, capsys, extra, message):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    with pytest.raises(SystemExit):
        parallel_bayes_gpu.main(["exc.csv", str(tmp_path / "out"), "obs.csv"] + extra)
    assert message in capsys.readouterr().err
    assert not (tmp_path / "out").exists()


def test_run_rejects_a_ladder_with_a_temperature(tmp_path):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    cfg = parallel_bayes_gpu.default_config()
    cfg["sim_flags"].update(sampler="ensemble", ladder=[1.0, 10.0], temperature=2.0)
    with pytest.raises(ValueError, match="exclude each other"):
        parallel_bayes_gpu.run("missing.csv", ["missing.csv"], [str(tmp_path / "out")], cfg=cfg)


def test_run_rejects_a_bad_ladder_before_reading_inputs(tmp_path):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    cfg = parallel_bayes_gpu.default_config()
    cfg["sim_flags"].update(sampler="ensemble", ladder=[2.0, 1.0])
    with pytest.raises(ValueError, match="strictly increasing"):
        parallel_bayes_gpu.run("missing.csv", ["missing.csv"], [str(tmp_path / "out")], cfg=cfg)


# ---------------------------------------------------------------------------------------------------------
# kernels against host mirrors
# ---------------------------------------------------------------------------------------------------------
def mirror_swap(X, lnl, K, first, W, temperatures, seed, step):
    """(X, lnl, flags, closest |ln u - r|) of trpl_tempered_swap on rows t n + i."""
    X, lnl = X.copy(), lnl.copy()
    n = X.shape[0] // K
    beta = 1.0 / np.asarray(temperatures, dtype=np.float64)
    flags = np.zeros((K - 1) * n, dtype=np.int32)
    closest = np.inf
    for i in range(n):
        for t in range(K - 1, 0, -1):
            h, c = t * n + i, (t - 1) * n + i
            lh, lc = (-np.inf if np.isnan(v) else float(v) for v in (lnl[h], lnl[c]))
            sw = False
            if not (lh == -np.inf and lc == -np.inf):
                r = (float(beta[t - 1]) - float(beta[t])) * (lh - lc)
                if r == np.inf:
                    sw = True
                elif r != -np.inf and r == r:
                    g = t * W + first + i
                    q = philox(g & MASK, g >> 32, step, 3, seed)
                    log_u = np.log(float((((q[0] << 32) | q[1]) >> 11) + 1) * 2.0 ** -53)
                    closest = min(closest, abs(log_u - r))
                    sw = bool(log_u < r)
            if sw:
                X[[h, c]] = X[[c, h]]
                lnl[[h, c]] = lnl[[c, h]]
            flags[c] = sw
    return X, lnl, flags, closest


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, 7])
def test_propose_matches_host_mirror_on_every_rung(flags):
    import torch
    from bayesian_inference_trpl_b200 import ensemble, tempering
    lo, hi = _engine_prior()
    rng = np.random.default_rng(13)
    K, W, first, n, a, seed, step = 3, 200, 107, 60, 2.0, 0x123456789AB, 17
    X = _prior_rows(K * n, lo, hi, rng)
    comp = _prior_rows(K * (W // 2), lo, hi, rng)
    for t, s in ensemble.override_sources(flags, 13).items():
        X[:, t], comp[:, t] = X[:, s], comp[:, s]
    comp_t = np.ascontiguousarray(np.concatenate([comp[t * (W // 2):(t + 1) * (W // 2)].T for t in range(K)]))
    Y, logq = tempering.propose(torch.from_numpy(X).cuda(), first, W, K, torch.from_numpy(comp_t).cuda(),
                                lo, hi, DO_LOG, flags, a, seed, step)
    Y, logq = Y.cpu().numpy(), logq.cpu().numpy()
    lin = ~DO_LOG.astype(bool)
    for t in range(K):
        rows = slice(t * n, (t + 1) * n)
        ref = mirror_propose(X[rows], t * W + first, W, comp[t * (W // 2):(t + 1) * (W // 2)], lo, hi, DO_LOG, flags,
                             a, seed, step)
        inside = np.array([r[2] for r in ref])
        assert 5 < inside.sum() < n - 5
        np.testing.assert_array_equal(np.isneginf(logq[rows]), ~inside)
        np.testing.assert_allclose(logq[rows][inside], [r[4] for r in ref if r[2]], rtol=1e-15, atol=0)
        Yref = np.array([r[3] for r in ref])
        np.testing.assert_array_equal(Y[rows][~inside], X[rows][~inside])
        np.testing.assert_array_equal(Y[rows][:, lin], Yref[:, lin])
        np.testing.assert_allclose(Y[rows][:, ~lin], Yref[:, ~lin], rtol=1e-13, atol=0)


@pytest.mark.gpu
def test_accept_matches_the_rule_on_every_rung():
    import torch
    from bayesian_inference_trpl_b200 import tempering
    rng = np.random.default_rng(14)
    T = np.array([1.0, 3.0, 10.0, INF])
    K, n, W, first, seed, step = 4, 300, 1000, 600, 99, 5
    lx = rng.normal(-10.0, 3.0, K * n)
    ly = rng.normal(-10.0, 3.0, K * n)
    q = rng.normal(0.0, 1.0, K * n)
    specials = [np.nan, -np.inf, np.inf]
    lx[rng.choice(K * n, 150, replace=False)] = rng.choice(specials[:2], 150)
    ly[rng.choice(K * n, 150, replace=False)] = rng.choice(specials, 150)
    q[rng.choice(K * n, 100, replace=False)] = -np.inf
    X = rng.normal(size=(K * n, 13))
    Y = rng.normal(size=(K * n, 13))
    Xd, lnl = torch.from_numpy(X).cuda(), torch.from_numpy(lx).cuda()
    acc = tempering.accept_(Xd, lnl, torch.from_numpy(Y).cuda(), torch.from_numpy(ly).cuda(),
                            torch.from_numpy(q).cuda(), first, W, T, seed, step).cpu().numpy().astype(bool)
    ex = np.where(np.isnan(lx), -np.inf, lx)
    ey = np.where(np.isnan(ly), -np.inf, ly)
    log_u = np.concatenate([mirror_log_u(t * W + first, n, seed, step) for t in range(K)])
    with np.errstate(invalid="ignore"):
        log_alpha = q + (ey - ex) / np.repeat(T, n)
    want = np.where(np.isneginf(q) | np.isneginf(ey), False, np.where(np.isneginf(ex), True, log_u < log_alpha))
    close = np.isfinite(ex) & np.isfinite(ey) & np.isfinite(q) & (np.abs(log_u - log_alpha) < 1e-12)
    np.testing.assert_array_equal(acc[~close], want[~close])
    for t in range(K):
        assert 30 < acc[t * n:(t + 1) * n].sum() < n - 30
    prior = slice(3 * n, 4 * n)                          # T = inf: the rule is ln u < log q for in-box proposals
    ok = np.isfinite(q[prior]) & np.isfinite(ey[prior]) & np.isfinite(ex[prior])
    np.testing.assert_array_equal(acc[prior][ok], (log_u[prior] < q[prior])[ok])
    Xg, lg = Xd.cpu().numpy(), lnl.cpu().numpy()
    np.testing.assert_array_equal(Xg[acc], Y[acc])
    np.testing.assert_array_equal(Xg[~acc], X[~acc])
    np.testing.assert_array_equal(lg[acc], ly[acc])
    np.testing.assert_array_equal(lg[~acc], lx[~acc])


@pytest.mark.gpu
def test_swap_matches_host_mirror():
    import torch
    from bayesian_inference_trpl_b200 import tempering
    rng = np.random.default_rng(15)
    T = np.array([1.0, 2.5, 7.0, INF])
    K, n, W, first, seed, step = 4, 250, 700, 350, 0xBEEF, 9
    lnl = rng.normal(-10.0, 3.0, K * n)
    lnl[rng.choice(K * n, 120, replace=False)] = rng.choice([np.nan, -np.inf], 120)
    lnl[:20] = lnl[n:n + 20] = -np.inf                  # both -inf between rungs 0 and 1
    lnl[n + 20:n + 30] = np.nan                          # NaN beside finite
    lnl[3 * n + 30:3 * n + 40] = -np.inf                 # the prior rung at -inf
    X = rng.normal(size=(K * n, 13))
    Xd, ld = torch.from_numpy(X).cuda(), torch.from_numpy(lnl).cuda()
    sw = tempering.swap_(Xd, ld, first, W, T, seed, step).cpu().numpy()
    Xm, lm, fm, closest = mirror_swap(X, lnl, K, first, W, T, seed, step)
    assert closest > 1e-12                               # no decision rests on the last bit of a log
    np.testing.assert_array_equal(sw, fm)
    np.testing.assert_array_equal(Xd.cpu().numpy(), Xm)
    np.testing.assert_array_equal(ld.cpu().numpy(), lm)  # raw lnL travels with its row, NaN included
    for t in range(K - 1):
        assert 20 < fm[t * n:(t + 1) * n].sum() < n - 20


# ---------------------------------------------------------------------------------------------------------
# the chain
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_one_rung_is_the_ensemble_sampler():
    from bayesian_inference_trpl_b200 import ensemble, tempering
    prob = _small_problem()
    lo, hi = _engine_prior()
    W, steps, flags, temp = 48, 6, 1, 2.0
    loglik = ensemble.solver_loglik(prob)
    X0 = ensemble.initial_walkers(W, lo, hi, DO_LOG, seed=5, override_flags=flags)
    np.testing.assert_array_equal(
        tempering.initial_walkers(W, 1, lo, hi, DO_LOG, seed=5, override_flags=flags).cpu().numpy(), X0.cpu().numpy())
    one = ensemble.sample(X0, loglik, lo, hi, DO_LOG, steps, override_flags=flags, temperature=temp, seed=5)
    pt = tempering.sample(X0, loglik, lo, hi, DO_LOG, steps, [temp], override_flags=flags, seed=5)
    assert pt.lnl.shape == (steps + 1, 1, W) and pt.acceptance.shape == (steps, 1)
    assert pt.swap_acceptance.shape == (steps, 0)
    np.testing.assert_array_equal(pt.X.cpu().numpy(), one.X.cpu().numpy())
    np.testing.assert_array_equal(pt.lnl[:, 0].cpu().numpy(), one.lnl.cpu().numpy())
    np.testing.assert_array_equal(pt.acceptance[:, 0].cpu().numpy(), one.acceptance.cpu().numpy())


def _same_chain_on_ranks(W, K, T, steps, seed, loglik, lo, hi, dl, worlds):
    """tempering.sample on 1 rank, then on `world` in-process ranks for each world: every rank's chain equals
    the one-rank chain bit for bit.  The barrier times out, so a rank that skips a collective fails the test
    instead of hanging it."""
    import torch
    from bayesian_inference_trpl_b200 import tempering
    one = tempering.sample(tempering.initial_walkers(W, K, lo, hi, dl, seed), loglik, lo, hi, dl, steps, T, seed=seed)
    for world in worlds:
        board = {"slots": [None] * world, "barrier": threading.Barrier(world, timeout=120)}
        results, errors = [None] * world, []

        def rank_main(r):
            try:
                torch.cuda.set_device(0)
                X0 = tempering.initial_walkers(W, K, lo, hi, dl, seed, rank=r, world=world)
                results[r] = tempering.sample(X0, loglik, lo, hi, dl, steps, T, n_walkers=W, seed=seed,
                                              exchange=_ThreadExchange(r, world, board))
                torch.cuda.synchronize()
            except Exception as e:                      # pragma: no cover - reported below
                errors.append(e)
                board["barrier"].abort()

        threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors, errors
        for res in results:
            for got, want in zip(res[:4], one[:4]):
                np.testing.assert_array_equal(got.cpu().numpy(), want.cpu().numpy())
    return one


@pytest.mark.gpu
def test_tempered_chain_is_the_same_for_any_number_of_ranks():
    """W = 26, K = 3: halves of 13 walkers per rung, shards of 7+6 and 4+3+3+3."""
    from bayesian_inference_trpl_b200 import ensemble
    lo, hi = _engine_prior()
    one = _same_chain_on_ranks(26, 3, [1.0, 30.0, INF], 5, 23, ensemble.solver_loglik(_small_problem()), lo, hi,
                               DO_LOG, (2, 4))
    assert float(one.swap_acceptance.sum()) > 0


@pytest.mark.gpu
def test_tempered_chain_with_ranks_that_hold_no_walkers():
    """W = 6 on the d = 3 Gaussian below: halves of 3 walkers per rung, so 4 ranks hold 1+1+1+0 and 8 ranks
    1+1+1+0+0+0+0+0 of each half.  The empty ranks still take part in every gather."""
    one = _same_chain_on_ranks(6, 3, [1.0, 4.0, INF], 12, 41, _gauss_loglik, G_LO, G_HI, G_LOG, (4, 8))
    assert float(one.acceptance.sum()) > 0


# d = 3 Gaussian (column 3 fixed) well inside a box whose half-width is 10x the hottest finite rung's width
G_MEAN = np.array([1.0, -2.0, 3.0])
G_SIGMA = np.array([1.0, 0.5, 2.0])
G_LADDER = np.array([1.0, 2.5, 6.25, INF])
G_HALF = 30.0 * G_SIGMA                                 # >= 10 sqrt(6.25) sigma
G_SHIFT = 5.0 * G_SIGMA                                 # box centre - mean
G_LO = np.append(G_MEAN + G_SHIFT - G_HALF, 7.0)
G_HI = np.append(G_MEAN + G_SHIFT + G_HALF, 7.0)
G_LOG = np.zeros(4, dtype=np.int32)


def _gauss_loglik(Y):
    import torch
    z = (Y[:, :3] - torch.from_numpy(G_MEAN).to(Y.device)) / torch.from_numpy(G_SIGMA).to(Y.device)
    return -0.5 * (z * z).sum(dim=1)


@pytest.mark.gpu
def test_every_rung_samples_its_tempered_gaussian():
    from bayesian_inference_trpl_b200 import tempering
    W, steps, seed = 4096, 800, 31
    K = G_LADDER.shape[0]
    ch = tempering.sample(tempering.initial_walkers(W, K, G_LO, G_HI, G_LOG, seed), _gauss_loglik, G_LO, G_HI,
                          G_LOG, steps, G_LADDER, seed=seed)
    assert ch.X.shape == (steps + 1, W, 4) and ch.lnl.shape == (steps + 1, K, W)
    assert ch.acceptance.shape == (steps, K) and ch.swap_acceptance.shape == (steps, K - 1)
    final = ch.lnl[-1].cpu().numpy()
    np.testing.assert_array_equal(final[0], _gauss_loglik(ch.X[-1]).cpu().numpy())
    assert (ch.X[..., 3] == 7.0).all()
    se = final.std(axis=1, ddof=1) / np.sqrt(W)
    want = -3.0 * G_LADDER / 2.0
    m2 = (2 * G_HALF) ** 2 / 12.0 + G_SHIFT ** 2        # the box's second moment about the mean
    want[-1] = -0.5 * float(np.sum(m2 / G_SIGMA ** 2))
    assert (np.abs(final.mean(axis=1) - want) < 5 * se).all(), (final.mean(axis=1), want, se)
    ev = tempering.log_evidence(ch.lnl, G_LADDER, burn=steps)
    np.testing.assert_allclose(ev.mean_lnl, final.mean(axis=1), rtol=1e-12)
    beta = 1.0 / G_LADDER
    weights = np.array([tempering._trapezoid(beta, e) for e in np.eye(K)])
    ref = tempering._trapezoid(beta, want)
    assert abs(ev.lnZ - ref) < 5 * np.sqrt(np.sum((weights * se) ** 2)), (ev.lnZ, ref)
    assert not ev.extrapolated
    acc = ch.acceptance[steps // 2:].mean(dim=0).cpu().numpy()
    assert (acc > 0.1).all(), acc


# 2-D mixture of two narrow Gaussians with weights 0.25 (x0 < 0) and 0.75 (x0 > 0) in a wide box
M_LO, M_HI = np.array([-10.0, -10.0]), np.array([10.0, 10.0])


def _mixture_loglik(Y):
    import torch
    s2 = 0.5 ** 2
    a = np.log(0.25) - 0.5 * ((Y[:, 0] + 4.0) ** 2 + Y[:, 1] ** 2) / s2
    b = np.log(0.75) - 0.5 * ((Y[:, 0] - 4.0) ** 2 + Y[:, 1] ** 2) / s2
    return torch.logaddexp(a, b)


@pytest.mark.gpu
def test_two_modes_get_their_weights():
    from bayesian_inference_trpl_b200 import ensemble, tempering
    W, steps, seed = 1024, 600, 8
    T = tempering.geometric_ladder(8, 300.0)
    dl = np.zeros(2, dtype=np.int32)
    ch = tempering.sample(tempering.initial_walkers(W, 8, M_LO, M_HI, dl, seed), _mixture_loglik, M_LO, M_HI, dl,
                          steps, T, seed=seed)
    share = float((ch.X[steps // 2:, :, 0] > 0).double().mean())
    se = np.sqrt(0.75 * 0.25 / W)                       # of one step; the mean over steps varies less
    assert abs(share - 0.75) < 5 * se, share
    swaps = ch.swap_acceptance[steps // 2:].mean(dim=0).cpu().numpy()
    assert (swaps > 0.05).all(), swaps
    plain = ensemble.sample(ensemble.initial_walkers(W, M_LO, M_HI, dl, seed), _mixture_loglik, M_LO, M_HI, dl, steps,
                            seed=seed)
    plain_share = float((plain.X[steps // 2:, :, 0] > 0).double().mean())
    assert abs(plain_share - 0.75) > 0.1, plain_share


# ---------------------------------------------------------------------------------------------------------
# command line
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cli_writes_the_tempered_chain(tmp_path):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    from test_nccl_exchange import _write_inputs
    exc, obs = _write_inputs(tmp_path)
    outs = {k: str(tmp_path / k) for k in ("TORCH", "CABI")}
    ladder = ["--ladder", "1", "10", "inf"]
    parallel_bayes_gpu.main(_cli_args(exc, obs, outs["TORCH"], ladder))
    parallel_bayes_gpu.main(_cli_args(exc, obs, outs["CABI"], ladder + ["--exchange", "cabi"]))
    files = {}
    for k, out in outs.items():
        b = os.path.join(out, os.path.basename(out))
        files[k] = _mcmc(out) + [np.load(b + "_MCMC_PT_P.npy")]
        with open(b + "_MCMC_PT.json") as fh:
            files[k].append(json.load(fh))
    X, Pl, PT, info = files["TORCH"]
    assert X.shape == (6, 32, 13) and Pl.shape == (6, 32) and PT.shape == (6, 3, 32)
    np.testing.assert_array_equal(Pl, PT[:, 0])
    cfg = parallel_bayes_gpu.default_config()
    lo, hi = cfg["minX"].astype(float), cfg["maxX"].astype(float)
    assert ((X >= lo * (1 - 1e-12)) & (X <= hi * (1 + 1e-12))).all()
    assert info["temperatures"] == [1.0, 10.0, "inf"] and info["prior_rung"] is True and info["burn"] == 2
    assert np.isfinite(info["log_evidence"]) and len(info["mean_lnl"]) == 3 and len(info["swap_acceptance"]) == 2
    assert len(info["acceptance"]) == 3 and info["nonfinite_lnl"] == int((~np.isfinite(PT)).sum())
    for a, b in zip(files["CABI"][:3], (X, Pl, PT)):
        np.testing.assert_array_equal(a, b)
    assert files["CABI"][3] == info
