"""CPU-only checks of the host side: observation bracketing, the bayeslib / bayes_io mirrors, and the
multi-rank plumbing (gloo)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import DO_LOG, GOLDEN, MAXX, MINX, UC, golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "bayesian_inference_trpl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no CPU fallback", ""), f


def test_obs_prepare_matches_searchsorted_rule():
    import bayesian_inference_trpl_b200 as trpl
    lib = trpl._lib.lib()
    Time, T = 7.5, 300
    grid = np.linspace(0, Time, T + 1)
    rng = np.random.default_rng(0)
    times = np.sort(np.concatenate([grid[::7], rng.uniform(0, Time, 50), [0.0, Time]]))
    n = len(times)
    hi = np.empty(n, np.int32); whi = np.empty(n); wlo = np.empty(n)
    rc = lib.trpl_obs_prepare(times.ctypes.data, n, Time, T, hi.ctypes.data, whi.ctypes.data,
                              wlo.ctypes.data)
    ref_hi = np.clip(np.searchsorted(grid, times), 1, T)
    np.testing.assert_array_equal(hi, ref_hi)
    assert rc == ref_hi.max()
    span = grid[ref_hi] - grid[ref_hi - 1]
    np.testing.assert_allclose(whi, (times - grid[ref_hi - 1]) / span, rtol=0, atol=1e-13)
    np.testing.assert_allclose(wlo, (grid[ref_hi] - times) / span, rtol=0, atol=1e-13)
    bad = np.array([0.0, Time * 1.01])
    assert lib.trpl_obs_prepare(bad.ctypes.data, 2, Time, T, hi.ctypes.data, whi.ctypes.data,
                                wlo.ctypes.data) < 0
    unsorted = np.array([1.0, 0.5])
    assert lib.trpl_obs_prepare(unsorted.ctypes.data, 2, Time, T, hi.ctypes.data,
                                whi.ctypes.data, wlo.ctypes.data) < 0


def test_interpolate_rows_matches_scipy_griddata():
    from scipy.interpolate import griddata
    from bayesian_inference_trpl_b200.bayeslib import interpolate_rows
    from oracle.oracle import interp_linear
    rng = np.random.default_rng(1)
    grid = np.linspace(0, 5, 201)
    rows = rng.normal(size=(4, 201)).astype(np.float32)
    times = np.sort(np.concatenate([grid[::9], rng.uniform(0, 5, 30)]))
    mine = interpolate_rows(grid, rows, times)
    orc = interp_linear(grid, rows, times)
    for i in range(4):
        ref = griddata(grid, rows[i], times)
        np.testing.assert_allclose(mine[i], ref, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(orc[i], ref, rtol=1e-12, atol=1e-13)


def test_make_grid_reproduces_reference_sample_matrix():
    """Seeded draw == X of the reference's bayeslib.bayes run recorded in the golden file."""
    path = os.path.join(GOLDEN, "cudasim_bayes.npz")
    if not os.path.exists(path):
        pytest.skip("golden not generated")
    from bayesian_inference_trpl_b200 import bayeslib
    g = golden("cudasim_bayes.npz")
    flags = {"override_equal_auger": False, "override_equal_mu": False, "override_equal_s": True,
             "random_sample": True, "num_points": len(g["X"])}
    np.random.seed(42)
    N, P, X = bayeslib.make_grid(np.array([0]), None, 1, g["minX"], g["maxX"], g["do_log"], flags)
    np.testing.assert_array_equal(X, g["X"])
    assert P.shape == (1, len(X)) and not P.any()
    np.testing.assert_array_equal(N, np.arange(len(X)))


def test_random_grid_bounds_and_fixed_columns():
    from bayesian_inference_trpl_b200 import bayeslib
    np.random.seed(0)
    X = bayeslib.random_grid(MINX * UC, MAXX * UC, DO_LOG, 1000)
    lo, hi = MINX * UC, MAXX * UC
    assert ((X >= lo - 1e-300) & (X <= hi * (1 + 1e-12))).all()
    assert (X[:, 0] == lo[0]).all() and (X[:, 11] == lo[11]).all() and (X[:, 12] == 0).all()


def test_bayes_io_roundtrip(tmp_path):
    from bayesian_inference_trpl_b200 import bayes_io
    t = [np.arange(0, 5) * 0.025, np.arange(0, 7) * 0.025]
    pl = [np.array([5., 4., 3., 2., 1.]) * 1e-7, np.array([9., 8., 7., 6., 5., 4., 3.]) * 1e-6]
    path = str(tmp_path / "obs.csv")
    bayes_io.write_observations(path, t, pl)
    flags = {"time_cutoff": 0.126, "select_obs_sets": None, "noise_level": None}
    e = bayes_io.get_data([path], flags, {"log_pl": True, "self_normalize": False})
    assert len(e) == 1 and len(e[0][0]) == 2
    np.testing.assert_allclose(e[0][0][0], t[0])
    np.testing.assert_allclose(e[0][1][0], np.log10(pl[0]), rtol=1e-9)
    assert len(e[0][0][1]) == 6                      # 0.15 ns cut off
    np.testing.assert_allclose(e[0][2][1], 1e14 * 1e-23 / pl[1][:6] / 2.3, rtol=1e-9)
    e2 = bayes_io.get_data([path], {"time_cutoff": None, "select_obs_sets": [1], "noise_level": None},
                           {"log_pl": False, "self_normalize": True})
    np.testing.assert_allclose(e2[0][1][0], pl[1] / pl[1].max(), rtol=1e-9)
    exc = str(tmp_path / "exc.csv")
    with open(exc, "w") as fh:
        fh.write("1E+16,2E+16,\n\n3E+16,4E+16,\n")
    ini = bayes_io.get_initpoints(exc, {"select_obs_sets": None})
    np.testing.assert_allclose(ini, np.array([[1e-5, 2e-5], [3e-5, 4e-5]]))
    out = str(tmp_path / "res" / "RUN1")
    os.makedirs(os.path.dirname(out))
    bayes_io.export(out, np.arange(3.0), np.ones((3, 13)))
    assert np.load(os.path.join(out, "RUN1_BAYRAN_P.npy")).shape == (3,)
    assert np.load(os.path.join(out, "RUN1_BAYRAN_X.npy")).shape == (3, 13)


def test_shard_bounds_cover_everything():
    from bayesian_inference_trpl_b200.distributed import shard_bounds
    for n in (0, 1, 7, 8, 1000003):
        for w in (1, 2, 3, 8):
            b = [shard_bounds(n, r, w) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            assert max(hi - lo for lo, hi in b) - min(hi - lo for lo, hi in b) <= 1


_WORKER = r"""
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
from bayesian_inference_trpl_b200 import distributed as D
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
rng = np.random.default_rng(5)
full = rng.normal(-800, 300, (2, 1001)); full[0, 17] = np.nan
lo, hi = D.shard_bounds(full.shape[1], rank, world)
local = torch.from_numpy(full[:, lo:hi].copy())
got = D.gather_rows(local, full.shape[1])
assert np.array_equal(got.numpy(), full, equal_nan=True)
# shard-local (max, sum exp) pairs, computed here with torch (the CUDA kernel is tested on the GPU)
m = torch.from_numpy(np.nanmax(full[:, lo:hi], axis=1))
s = torch.from_numpy(np.nansum(np.exp(full[:, lo:hi] - m.numpy()[:, None]), axis=1))
lse = D.global_logsumexp(torch.stack([m, s], dim=-1))
mm = np.nanmax(full, axis=1)
ref = mm + np.log(np.nansum(np.exp(full - mm[:, None]), axis=1))
assert np.allclose(lse.numpy(), ref, rtol=1e-13), (lse, ref)
w = D.normalize_posterior(got, lse[:, None])
assert np.allclose(np.nansum(w.numpy(), axis=1), 1.0, rtol=1e-12)
# block-cyclic merge (reference layout: zeros outside own blocks)
P = np.zeros((1, 10)); G = 2
for b in range(rank * G, 10, world * G): P[0, b:b + G] = np.arange(b, min(b + G, 10)) + 1.0
tot = D.merge_block_cyclic(P.copy())
assert np.array_equal(np.asarray(tot), np.arange(10)[None] + 1.0)
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_two_rank_gloo_gather_and_logsumexp(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT})
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1",
                   MASTER_PORT="29581")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        out, _ = p.communicate(timeout=240)
        assert p.returncode == 0, out.decode()


def test_bayes_io_matches_reference_reader():
    """bayes_io.get_data / get_initpoints vs the reference's own readers on the same files
    (golden made by tests/golden/make_io_golden.py)."""
    from bayesian_inference_trpl_b200 import bayes_io
    g = golden("io_golden.npz")
    obs, exc = os.path.join(GOLDEN, "io_obs.csv"), os.path.join(GOLDEN, "io_exc.csv")
    cases = {"log": ({"time_cutoff": None, "select_obs_sets": None, "noise_level": None},
                     {"log_pl": True, "self_normalize": False}),
             "cut_sel": ({"time_cutoff": 0.126, "select_obs_sets": [0, 2], "noise_level": None},
                         {"log_pl": True, "self_normalize": False}),
             "norm_lin": ({"time_cutoff": None, "select_obs_sets": None, "noise_level": None},
                          {"log_pl": False, "self_normalize": True})}
    for name, (ic, sf) in cases.items():
        e = bayes_io.get_data([obs], ic, sf, scale_f=1e-23)[0]
        assert len(e[0]) == int(g[name + "_n"])
        for k, part in enumerate(("t", "pl", "unc")):
            for c in range(len(e[0])):
                np.testing.assert_array_equal(np.asarray(e[k][c]), g["%s_%s%d" % (name, part, c)])
        np.testing.assert_array_equal(bayes_io.get_initpoints(exc, ic), g[name + "_ini"])


def test_no_cpu_fallback_without_a_gpu():
    """On a machine without CUDA every product entry point raises instead of computing on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("this check is for GPU-less machines")
    import bayesian_inference_trpl_b200 as trpl
    pl = np.zeros((1, 5))
    with pytest.raises(trpl.TrplError):
        trpl.pvSim(pl, None, None, None, np.ones((1, 12)), [100.0, 1.0, 8, 4, 1, (0,), 7, 100], np.ones(8),
                   (8,), 1, 1, init_mode="points")
    with pytest.raises(trpl.TrplError):
        trpl.fastlog(np.ones((2, 2)), 1e-300)
    with pytest.raises(trpl.TrplError):
        trpl.prob(np.zeros(2), np.ones((2, 3)), np.ones(3), np.ones(3), np.zeros(2))
    with pytest.raises((trpl.TrplError, RuntimeError)):
        trpl.bayeslib.simulate(trpl.pvSim, [], np.zeros((1, 1)), np.ones((1, 13)), [None], [None], 1,
                               [100.0, 1.0, 8, 4, 1, (0,), 7, 100], np.ones((1, 8)),
                               {"load_PL_from_file": False, "log_pl": True, "self_normalize": False},
                               {"has_GPU": False, "sims_per_gpu": 1, "num_gpus": 1}, 0,
                               np.zeros(1), np.zeros(1), np.zeros(1))


def test_slurm_array_mode_rank_world_and_owned_columns(monkeypatch):
    """ADVICE r1: under SLURM arrays the task count must be known or checked, and columns a task does
    not own must not read as lnL = 0 (the best possible likelihood)."""
    from bayesian_inference_trpl_b200 import bayeslib
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.setenv("SLURM_ARRAY_TASK_ID", "2")
    monkeypatch.delenv("SLURM_ARRAY_TASK_COUNT", raising=False)
    assert bayeslib.rank_and_world() == (2, None)
    monkeypatch.setenv("SLURM_ARRAY_TASK_COUNT", "4")
    assert bayeslib.rank_and_world() == (2, 4)
    info = {"sims_per_gpu": 3, "num_gpus": 4}
    masks = [bayeslib.owned_columns(29, info, r) for r in range(4)]
    assert np.array_equal(np.sum(masks, axis=0), np.ones(29, dtype=int))      # a partition of the columns
    assert masks[2][6:9].all() and not masks[2][:6].any() and masks[2][18:21].all()


def test_merge_task_exports(tmp_path):
    from bayesian_inference_trpl_b200 import bayes_io, bayeslib, parallel_bayes_gpu as entry
    rng = np.random.default_rng(0)
    S = 23
    X = rng.normal(size=(S, 13))
    P = rng.normal(size=S)
    info = {"sims_per_gpu": 4, "num_gpus": 3}
    out = str(tmp_path / "run")
    for k in range(3):
        mine = bayeslib.owned_columns(S, info, k)
        bayes_io.export("%s_task%d" % (out, k), np.where(mine, P, np.nan), X)
    Pm, Xm = entry.merge_task_exports(out, 3)
    np.testing.assert_array_equal(Pm, P)
    np.testing.assert_array_equal(Xm, X)
    base = os.path.basename(out)
    np.testing.assert_array_equal(np.load(os.path.join(out, base + "_BAYRAN_P.npy")), P)


def test_vectorised_observation_reader_handles_the_reference_format_corners(tmp_path):
    """One-pass reader: END row, blank lines, CRLF, a return to t=0 starts a new curve, ragged rows."""
    from bayesian_inference_trpl_b200 import bayes_io
    p = tmp_path / "o.csv"
    p.write_text("0,1.5E+20,1E14\r\n0.025,1.25E+20,1E14\r\n\r\n0.05,1.0E+20,1E14\n0,3E+19,1E14\n0.025,2E+19,1E14\nEND\n9,9,9\n")
    e = bayes_io.get_data([str(p)], {"time_cutoff": None, "select_obs_sets": None, "noise_level": None},
                          {"log_pl": False, "self_normalize": False}, scale_f=1.0)[0]
    assert [len(t) for t in e[0]] == [3, 2]
    np.testing.assert_array_equal(e[0][0], [0, 0.025, 0.05])
    np.testing.assert_array_equal(e[1][1], [3e19, 2e19])
    q = tmp_path / "ragged.csv"
    q.write_text("0,1,2,extra\n1,3,4\nEND\n")
    e = bayes_io.get_data([str(q)], {"time_cutoff": None, "select_obs_sets": None, "noise_level": None},
                          {"log_pl": False, "self_normalize": False}, scale_f=1.0)[0]
    np.testing.assert_array_equal(e[1][0], [1, 3])


def test_export_from_device_writes_valid_npy_on_cpu_tensors(tmp_path):
    import torch
    from bayesian_inference_trpl_b200 import bayes_io
    P = torch.arange(1000, dtype=torch.float64) * -0.5
    X = torch.arange(13000, dtype=torch.float64).reshape(1000, 13)
    out = str(tmp_path / "DEV")
    bayes_io.export_from_device(out, P, X, chunk_rows=128)
    np.testing.assert_array_equal(np.load(os.path.join(out, "DEV_BAYRAN_P.npy")), P.numpy())
    np.testing.assert_array_equal(np.load(os.path.join(out, "DEV_BAYRAN_X.npy")), X.numpy())
