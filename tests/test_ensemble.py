"""The ensemble sampler (ensemble.py, include/trpl_b200_ensemble.h): the binding agrees with the header, bad
arguments are refused before the device is entered, and the host rules (free columns, halves, shards) hold;
on a GPU the two kernels agree with a host mirror of their Philox draws and rules, the chain samples a known
target, its bookkeeping agrees with the solver, it does not depend on the number of ranks, and the command
line writes the chain."""
import ctypes
import os
import re
import subprocess
import sys
import threading
from fractions import Fraction

import numpy as np
import pytest

from helpers import DO_LOG, MAXX, MINX, TRUTH, UC, power_scan_excitations

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "trpl_b200_ensemble.h")

EINVAL, ENODEVICE = -1, -4
P = ctypes.c_void_p(16)          # placeholder device pointer: no case below dereferences it


@pytest.fixture(scope="module")
def elib():
    import bayesian_inference_trpl_b200 as trpl
    trpl.build()
    return trpl.ensemble.lib()


def _header():
    src = re.sub(r"/\*.*?\*/", " ", open(HEADER).read(), flags=re.S)
    src = re.sub(r"#.*", " ", src)
    funcs = {}
    for m in re.finditer(r"([\w\s\*]+?)\b(trpl_\w+)\s*\(([^)]*)\)\s*;", src):
        params = [" ".join(p.split()) for p in m.group(3).split(",")]
        params = [re.sub(r"\s*\b\w+$", "", p) for p in params]
        funcs[m.group(2)] = (" ".join(m.group(1).split()), params)
    return funcs


def _ctype(ctype):
    if ctype.endswith("*"):
        return ctypes.c_void_p
    return {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64,
            "uint32_t": ctypes.c_uint32, "double": ctypes.c_double}[ctype]


def test_binding_matches_header(elib):
    from bayesian_inference_trpl_b200 import _lib, ensemble
    funcs = _header()
    assert list(funcs) == ensemble.EXPORTS == ["trpl_stretch_propose", "trpl_stretch_accept"]
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name, (ret, params) in funcs.items():
        assert hasattr(raw, name), name
        restype, argtypes = ensemble._SIGNATURES[name]
        assert restype is _ctype(ret), name
        assert [_ctype(p) for p in params] == argtypes, name
        fn = getattr(elib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name
    assert set(_lib.EXPORTS).isdisjoint(funcs)          # trpl_b200.h keeps its own table


def _bounds(ncol=13):
    lo, hi = np.zeros(17), np.ones(17)
    lo[0] = hi[0] = 0.5                                 # one fixed column: d = ncol - 1
    return lo, hi, np.zeros(17, dtype=np.int32)


def _propose(lib, d_x=P, n=4, ncol=13, a=2.0, first=0, W=32, device=-1):
    lo, hi, dl = _bounds()
    return lib.trpl_stretch_propose(d_x, n, 17, first, W, P, 64, lo.ctypes.data, hi.ctypes.data, dl.ctypes.data,
                                    ncol, 0, a, 1, 0, P, 17, P, device, None)


def _accept(lib, d_lnl=P, n=4, ncol=13, first=0, W=32, temperature=1.0, device=-1):
    return lib.trpl_stretch_accept(P, n, 17, first, W, ncol, d_lnl, P, 17, P, P, temperature, 1, 0, None, device, None)


def test_return_code_contract(elib):
    cases = [
        (_propose(elib, d_x=None), EINVAL),
        (_propose(elib, n=-1), EINVAL),
        (_propose(elib, ncol=17), EINVAL),
        (_propose(elib, a=1.0), EINVAL),
        (_propose(elib, a=float("nan")), EINVAL),
        (_propose(elib, W=31), EINVAL),                 # odd
        (_propose(elib, W=22), EINVAL),                 # fewer than 2 x 12 free columns
        (_propose(elib, W=24, n=12), ENODEVICE),
        (_propose(elib, first=14), EINVAL),             # crosses from half A into half B
        (_propose(elib, first=29, n=4), EINVAL),        # past the last walker
        (_propose(elib), ENODEVICE),
        (_propose(elib, first=16, n=16), ENODEVICE),
        (_accept(elib, d_lnl=None), EINVAL),
        (_accept(elib, n=-1), EINVAL),
        (_accept(elib, ncol=17), EINVAL),
        (_accept(elib, W=31), EINVAL),
        (_accept(elib, W=0, n=0), EINVAL),
        (_accept(elib, first=14), EINVAL),
        (_accept(elib, temperature=0.0), EINVAL),
        (_accept(elib), ENODEVICE),
    ]
    assert [rc for rc, _ in cases] == [want for _, want in cases]


def test_free_columns_and_walker_count():
    from bayesian_inference_trpl_b200 import ensemble
    lo, hi = MINX * UC, MAXX * UC
    # default prior: n0, lambda and mag_offset are fixed
    assert ensemble.free_columns(lo, hi).sum() == 10
    # override_equal_mu/s/auger: columns 2, 6, 8 follow 3, 5, 7
    assert list(np.flatnonzero(ensemble.free_columns(lo, hi, 7))) == [1, 3, 4, 5, 7, 9, 10]
    assert list(np.flatnonzero(ensemble.free_columns(lo, hi, 2))) == [1, 2, 3, 4, 5, 7, 8, 9, 10]
    assert ensemble.override_sources(7, 13) == {2: 3, 6: 5, 8: 7}
    assert ensemble.override_sources(7, 6) == {2: 3}    # a column the row does not have is not overridden
    ensemble.check_walkers(20, 10)
    for W, d in ((19, 1), (18, 10), (0, 0), (1, 0)):
        with pytest.raises(ValueError):
            ensemble.check_walkers(W, d)


@pytest.mark.parametrize("W", [2, 18, 64, 1001 * 2])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_halves_and_shards(W, world):
    from bayesian_inference_trpl_b200 import distributed, ensemble
    h = W // 2
    parts = [ensemble.local_rows(W, r, world) for r in range(world)]
    for k, base in ((0, 0), (1, h)):
        got = [i for p in parts for i in range(*p[k])]
        assert got == list(range(base, base + h))       # each half is split contiguously, in rank order
        for r, p in enumerate(parts):
            lo, hi = distributed.shard_bounds(h, r, world)
            assert p[k] == (base + lo, base + hi)


def test_cli_rejects_two_observation_files(tmp_path):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    with pytest.raises(ValueError, match="one observation file"):
        parallel_bayes_gpu.main(["exc.csv", str(tmp_path / "out"), "a.csv", "b.csv", "--sampler", "ensemble"])


# ---------------------------------------------------------------------------------------------------------
# host mirror of the kernels
# ---------------------------------------------------------------------------------------------------------
MASK = (1 << 32) - 1


def philox(c0, c1, c2, c3, key):
    """Philox4x32-10 (trpl_aux_kernels.cuh) on Python ints."""
    k0, k1 = key & MASK, key >> 32
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & MASK, (p0 >> 32) ^ c3 ^ k1, p0 & MASK
        k0, k1 = (k0 + 0x9E3779B9) & MASK, (k1 + 0xBB67AE85) & MASK
    return c0, c1, c2, c3


def fma(x, y, z):
    """Correctly rounded x*y + z."""
    return float(Fraction(x) * Fraction(y) + Fraction(z))


def mirror_propose(X, first, W, comp, lo, hi, dl, flags, a, seed, step):
    """(partner, z, inside, Y, logq) of trpl_stretch_propose; comp [W/2, ncol] rows."""
    from bayesian_inference_trpl_b200 import ensemble
    ncol = X.shape[1]
    src = {j: j for j in range(ncol)}
    src.update(ensemble.override_sources(flags, ncol))
    free = ensemble.free_columns(lo, hi, flags)
    d = int(free.sum())
    out = []
    for i, xk in enumerate(X):
        g = first + i
        r = philox(g & MASK, g >> 32, step, 1, seed)
        p = (((r[0] << 32) | r[1]) * (W // 2)) >> 64
        u = float(((r[2] << 32) | r[3]) >> 11) * 2.0 ** -53
        t = fma(a - 1.0, u, 1.0)
        z = t * t / a
        xp = comp[p]
        inside, y = True, xk.copy()
        for j in np.flatnonzero(free):
            if dl[j]:
                tp = np.log10(xp[j])
                v = fma(z, np.log10(xk[j]) - tp, tp)
                inside &= bool(np.log10(lo[j]) <= v <= np.log10(hi[j]))
                y[j] = 10.0 ** v
            else:
                v = fma(z, xk[j] - xp[j], xp[j])
                inside &= bool(lo[j] <= v <= hi[j])
                y[j] = v
        y = np.array([y[src[j]] for j in range(ncol)])
        out.append((p, z, inside, y if inside else xk.copy(), (d - 1) * np.log(z) if inside else -np.inf))
    return out


def mirror_log_u(first, n, seed, step):
    res = []
    for i in range(n):
        g = first + i
        r = philox(g & MASK, g >> 32, step, 2, seed)
        res.append(np.log(float((((r[0] << 32) | r[1]) >> 11) + 1) * 2.0 ** -53))
    return np.array(res)


def _engine_prior():
    lo, hi = MINX * UC, MAXX * UC
    lo[2:4] = 0.5 * UC[2]
    lo[12], hi[12] = -0.2, 0.2
    return lo, hi


def _prior_rows(n, lo, hi, rng):
    X = np.empty((n, 13))
    for j in range(13):
        if DO_LOG[j] and lo[j] != hi[j]:
            X[:, j] = 10 ** rng.uniform(np.log10(lo[j]), np.log10(hi[j]), n)
        else:
            X[:, j] = rng.uniform(lo[j], hi[j], n)
    return X


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, 7])
def test_propose_matches_host_mirror(flags):
    import torch
    from bayesian_inference_trpl_b200 import ensemble
    lo, hi = _engine_prior()
    rng = np.random.default_rng(3)
    W, first, n, a, seed, step = 200, 107, 60, 2.0, 0x123456789AB, 17
    X = _prior_rows(n, lo, hi, rng)
    comp = _prior_rows(W // 2, lo, hi, rng)
    for t, s in ensemble.override_sources(flags, 13).items():
        X[:, t], comp[:, t] = X[:, s], comp[:, s]
    Y, logq = ensemble.propose(torch.from_numpy(X).cuda(), first, W, torch.from_numpy(comp.T.copy()).cuda(),
                               lo, hi, DO_LOG, flags, a, seed, step)
    Y, logq = Y.cpu().numpy(), logq.cpu().numpy()
    ref = mirror_propose(X, first, W, comp, lo, hi, DO_LOG, flags, a, seed, step)
    inside = np.array([r[2] for r in ref])
    assert 5 < inside.sum() < n - 5                     # both kinds occur
    np.testing.assert_array_equal(np.isneginf(logq), ~inside)
    np.testing.assert_allclose(logq[inside], [r[4] for r in ref if r[2]], rtol=1e-15, atol=0)
    Yref = np.array([r[3] for r in ref])
    np.testing.assert_array_equal(Y[~inside], X[~inside])          # out of the box: the walker's own row
    lin = ~DO_LOG.astype(bool)
    np.testing.assert_array_equal(Y[:, lin], Yref[:, lin])         # partner and z equal, FMAs exact
    np.testing.assert_allclose(Y[:, ~lin], Yref[:, ~lin], rtol=1e-13, atol=0)   # log10/exp10 of the device
    fixed = lo == hi
    np.testing.assert_array_equal(Y[:, fixed], X[:, fixed])
    for t, s in ensemble.override_sources(flags, 13).items():
        np.testing.assert_array_equal(Y[:, t], Y[:, s])


@pytest.mark.gpu
def test_accept_matches_the_rule():
    import torch
    from bayesian_inference_trpl_b200 import ensemble
    rng = np.random.default_rng(4)
    n, W, first, T, seed, step = 400, 1000, 600, 3.0, 99, 5
    lx = rng.normal(-10.0, 3.0, n)
    ly = rng.normal(-10.0, 3.0, n)
    q = rng.normal(0.0, 1.0, n)
    specials = [np.nan, -np.inf, np.inf]
    lx[rng.choice(n, 60, replace=False)] = rng.choice(specials[:2], 60)
    ly[rng.choice(n, 60, replace=False)] = rng.choice(specials, 60)
    q[rng.choice(n, 40, replace=False)] = -np.inf
    X = rng.normal(size=(n, 13))
    Y = rng.normal(size=(n, 13))
    Xd, lnl = torch.from_numpy(X).cuda(), torch.from_numpy(lx).cuda()
    acc = ensemble.accept_(Xd, lnl, torch.from_numpy(Y).cuda(), torch.from_numpy(ly).cuda(),
                           torch.from_numpy(q).cuda(), first, W, T, seed, step).cpu().numpy().astype(bool)
    ex = np.where(np.isnan(lx), -np.inf, lx)
    ey = np.where(np.isnan(ly), -np.inf, ly)
    log_u = mirror_log_u(first, n, seed, step)
    with np.errstate(invalid="ignore"):
        log_alpha = q + (ey - ex) / T
    want = np.where(np.isneginf(q) | np.isneginf(ey), False, np.where(np.isneginf(ex), True, log_u < log_alpha))
    close = np.isfinite(ex) & np.isfinite(ey) & np.isfinite(q) & (np.abs(log_u - log_alpha) < 1e-12)
    np.testing.assert_array_equal(acc[~close], want[~close])
    assert 50 < acc.sum() < n - 50
    Xg, lg = Xd.cpu().numpy(), lnl.cpu().numpy()
    np.testing.assert_array_equal(Xg[acc], Y[acc])
    np.testing.assert_array_equal(Xg[~acc], X[~acc])
    np.testing.assert_array_equal(lg[acc], ly[acc])
    np.testing.assert_array_equal(lg[~acc], lx[~acc])               # NaN walkers keep their NaN


# ---------------------------------------------------------------------------------------------------------
# the chain
# ---------------------------------------------------------------------------------------------------------
GAUSS_LO = np.array([-10.0, 1e-3, 0.0, -5.0])
GAUSS_HI = np.array([12.0, 1e4, 20.0, 15.0])
GAUSS_LOG = np.array([0, 1, 0, 0])
GAUSS_MEAN = np.array([1.0, 0.5, 5.0])                # in (x0, log10 x1, x3)
GAUSS_COV = np.array([[1.0, 0.95 * 0.3, 0.0], [0.95 * 0.3, 0.09, 0.0], [0.0, 0.0, 1.0]])


def _gauss_loglik(Y):
    import torch
    prec = torch.from_numpy(np.linalg.inv(GAUSS_COV)).to(Y.device)
    z = torch.stack([Y[:, 0], torch.log10(Y[:, 1]), Y[:, 3]], dim=1) - torch.from_numpy(GAUSS_MEAN).to(Y.device)
    return -0.5 * ((z @ prec) * z).sum(dim=1)


@pytest.mark.gpu
def test_stationary_distribution_of_a_correlated_gaussian():
    """rho = 0.95 between a linear and a log-scaled column, well inside the box, column 2 overridden from 3:
    after burn-in the final ensemble has the target's mean and covariance within 5 standard errors."""
    import torch
    from bayesian_inference_trpl_b200 import ensemble
    W, steps = 4096, 1000
    X0 = ensemble.initial_walkers(W, GAUSS_LO, GAUSS_HI, GAUSS_LOG, seed=11, override_flags=1)
    ch = ensemble.sample(X0, _gauss_loglik, GAUSS_LO, GAUSS_HI, GAUSS_LOG, steps, override_flags=1, seed=11)
    assert ch.X.shape == (steps + 1, W, 4) and ch.lnl.shape == (steps + 1, W) and ch.acceptance.shape == (steps,)
    X = ch.X[-1].cpu().numpy()
    assert (X[:, 2] == X[:, 3]).all()
    T = np.stack([X[:, 0], np.log10(X[:, 1]), X[:, 3]], axis=1)
    mean_se = np.sqrt(np.diag(GAUSS_COV) / W)
    assert (np.abs(T.mean(axis=0) - GAUSS_MEAN) < 5 * mean_se).all(), (T.mean(axis=0), mean_se)
    cov = np.cov(T, rowvar=False)
    var = np.diag(GAUSS_COV)
    cov_se = np.sqrt((np.outer(var, var) + GAUSS_COV ** 2) / W)
    assert (np.abs(cov - GAUSS_COV) < 5 * cov_se).all(), (cov, cov_se)
    acc = float(ch.acceptance[steps // 2:].mean())
    assert 0.2 < acc < 0.8, acc
    torch.testing.assert_close(ch.lnl[-1], _gauss_loglik(ch.X[-1]), rtol=1e-12, atol=1e-12)


def _small_problem(T=200):
    from bayesian_inference_trpl_b200 import engine
    L, Time = 128, 0.025 * T
    inis = power_scan_excitations()
    import torch
    m = torch.from_numpy((TRUTH * UC)[None, :12].copy()).cuda()
    grid = np.linspace(0, Time, T + 1)
    pls = [engine.solve_pl(m, torch.from_numpy(inis[c]).cuda(), 2000.0, Time, L, T)[0][0].cpu().numpy()
           for c in range(3)]
    e_data = [([grid] * 3, [np.log10(p) for p in pls], [np.full(T + 1, 0.1)] * 3)]
    return engine.Problem([2000.0, Time, L, T, 1, (0,), 7, 10000], inis, e_data, device=0)


def _inside(X, lo, hi):
    lo_t = np.where(DO_LOG == 1, np.log10(np.where(lo > 0, lo, 1)), lo)
    hi_t = np.where(DO_LOG == 1, np.log10(np.where(hi > 0, hi, 1)), hi)
    with np.errstate(divide="ignore", invalid="ignore"):
        T = np.where(DO_LOG == 1, np.log10(X), X)
    return ((T >= lo_t - 1e-12 * np.abs(lo_t)) & (T <= hi_t + 1e-12 * np.abs(hi_t))).all()


@pytest.mark.gpu
def test_bookkeeping_with_the_solver():
    import torch
    from bayesian_inference_trpl_b200 import engine, ensemble
    prob = _small_problem()
    lo, hi = _engine_prior()
    W, steps, flags = 48, 8, 1
    X0 = ensemble.initial_walkers(W, lo, hi, DO_LOG, seed=5, override_flags=flags)
    ch = ensemble.sample(X0, ensemble.solver_loglik(prob), lo, hi, DO_LOG, steps, override_flags=flags, seed=5)
    X, lnl = ch.X.cpu().numpy(), ch.lnl.cpu().numpy()
    assert _inside(X, lo, hi)
    assert (X[..., 2] == X[..., 3]).all()
    assert (X[..., lo == hi] == lo[lo == hi]).all()
    again, _, _ = engine.solve_loglik(ch.X.reshape(-1, 13).contiguous(), prob)
    np.testing.assert_array_equal(again[0].cpu().numpy().reshape(steps + 1, W), lnl)
    assert np.nanmedian(lnl[-1]) > np.nanmedian(lnl[0])
    assert float(ch.acceptance.sum()) > 0


class _ThreadExchange:
    """In-process exchange of `world` threads on one GPU: gather_rows concatenates every thread's shard.  All
    threads enqueue on the device's default stream, so a shard is complete before a reader's kernels run."""

    def __init__(self, rank, world, board):
        self.rank, self.world, self.board = rank, world, board

    def rank_world(self):
        return self.rank, self.world

    def gather_rows(self, local, n_total):
        b = self.board
        b["slots"][self.rank] = local
        b["barrier"].wait()
        out = __import__("torch").cat([b["slots"][r] for r in range(self.world)], dim=-1)
        b["barrier"].wait()
        assert out.shape[-1] == n_total
        return out


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_chain_is_the_same_for_any_number_of_ranks(world):
    """W = 26: halves of 13 walkers, shards of 7+6 (two ranks) and 4+3+3+3 (four ranks)."""
    import torch
    from bayesian_inference_trpl_b200 import ensemble
    prob = _small_problem()
    loglik = ensemble.solver_loglik(prob)
    lo, hi = _engine_prior()
    W, steps, seed = 26, 6, 21
    one = ensemble.sample(ensemble.initial_walkers(W, lo, hi, DO_LOG, seed), loglik, lo, hi, DO_LOG, steps, seed=seed)
    board = {"slots": [None] * world, "barrier": threading.Barrier(world)}
    results, errors = [None] * world, []

    def rank_main(r):
        try:
            torch.cuda.set_device(0)
            X0 = ensemble.initial_walkers(W, lo, hi, DO_LOG, seed, rank=r, world=world)
            results[r] = ensemble.sample(X0, loglik, lo, hi, DO_LOG, steps, n_walkers=W, seed=seed,
                                         exchange=_ThreadExchange(r, world, board))
            torch.cuda.synchronize()
        except Exception as e:                          # pragma: no cover - reported below
            errors.append(e)
            board["barrier"].abort()

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for res in results:
        for got, want in zip(res, one):
            np.testing.assert_array_equal(got.cpu().numpy(), want.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------
# command line
# ---------------------------------------------------------------------------------------------------------
def _cli_args(exc, obs, out, extra=()):
    return [exc, out, obs, "--sampler", "ensemble", "--walkers", "32", "--steps", "5", "--length", "2000",
            "--time-steps", "240", "--final-time", str(0.025 * 240)] + list(extra)


def _mcmc(out):
    b = os.path.basename(out)
    return [np.load(os.path.join(out, "%s_MCMC_%s.npy" % (b, k))) for k in "XP"]


@pytest.mark.gpu
def test_cli_writes_the_chain(tmp_path):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    from test_nccl_exchange import _write_inputs
    exc, obs = _write_inputs(tmp_path)
    outs = {k: str(tmp_path / k) for k in ("TORCH", "CABI")}
    parallel_bayes_gpu.main(_cli_args(exc, obs, outs["TORCH"]))
    parallel_bayes_gpu.main(_cli_args(exc, obs, outs["CABI"], ["--exchange", "cabi"]))
    X, Pl = _mcmc(outs["TORCH"])
    assert X.shape == (6, 32, 13) and Pl.shape == (6, 32)
    cfg = parallel_bayes_gpu.default_config()
    lo, hi = cfg["minX"].astype(float), cfg["maxX"].astype(float)
    assert ((X >= lo * (1 - 1e-12)) & (X <= hi * (1 + 1e-12))).all()          # common units
    for a, b in zip(_mcmc(outs["CABI"]), (X, Pl)):
        np.testing.assert_array_equal(a, b)


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_ngpu() < 2, reason="needs at least 2 GPUs")
def test_two_ranks_under_torchrun_match_one_rank(tmp_path):
    from test_nccl_exchange import _write_inputs
    exc, obs = _write_inputs(tmp_path)
    flags = ["-s"] if sys.flags.no_user_site else []
    base = [sys.executable] + flags + ["-m", "bayesian_inference_trpl_b200.parallel_bayes_gpu"]
    one, two = str(tmp_path / "ONE"), str(tmp_path / "TWO")
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    subprocess.run(base + _cli_args(exc, obs, one), cwd=ROOT, env=env, check=True, timeout=300)
    subprocess.run([sys.executable] + flags + ["-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2",
                    "-m", "bayesian_inference_trpl_b200.parallel_bayes_gpu"] + _cli_args(exc, obs, two),
                   cwd=ROOT, env=env, check=True, timeout=300)
    for a, b in zip(_mcmc(two), _mcmc(one)):
        np.testing.assert_array_equal(a, b)
