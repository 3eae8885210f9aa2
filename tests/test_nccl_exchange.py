"""The NCCL companion library libtrpl_b200_nccl.so and nccl.Communicator: the binding agrees with
include/trpl_b200_nccl.h, bad arguments are refused before the device is entered, only the companion
links NCCL; on one GPU the exchange is exact (one rank) and run(..., exchange=...) writes the same files
as the default path; on several GPUs, ranks in separate processes without torch.distributed agree with
the full table computed in one process."""
import ctypes
import os
import re
import subprocess
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "trpl_b200_nccl.h")

EINVAL, ENODEVICE = -1, -4
P = ctypes.c_void_p(16)          # placeholder pointer: no case below dereferences it


@pytest.fixture(scope="module")
def nlib():
    import bayesian_inference_trpl_b200 as trpl
    from bayesian_inference_trpl_b200 import nccl
    trpl.build()
    nccl.build()
    return nccl.lib()


def _header():
    """{name: (return type, [parameter types])} in header order and {TRPL_* define: value} of the C header
    (the parser of test_host_boundary, plus opaque struct typedefs)."""
    src = re.sub(r"/\*.*?\*/", " ", open(HEADER).read(), flags=re.S)
    defines = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(TRPL_\w+)\s+(-?\d+)\b", src)}
    src = re.sub(r"typedef struct\s+\w+\s+\w+\s*;", " ", src)
    src = re.sub(r"#.*", " ", src)
    funcs = {}
    for m in re.finditer(r"([\w\s\*]+?)\b(trpl_\w+)\s*\(([^)]*)\)\s*;", src):
        params = [" ".join(p.split()) for p in m.group(3).split(",")]
        params = [] if params == ["void"] else [re.sub(r"\s*\b\w+$", "", p) for p in params]
        funcs[m.group(2)] = (" ".join(m.group(1).split()), params)
    return funcs, defines


def _ctype(ctype):
    if ctype == "const char *":
        return ctypes.c_char_p
    if ctype.endswith("*"):
        return ctypes.c_void_p
    return {"int": ctypes.c_int, "int64_t": ctypes.c_int64}[ctype]


def test_binding_matches_header(nlib):
    from bayesian_inference_trpl_b200 import nccl
    funcs, defines = _header()
    assert list(funcs) == nccl.EXPORTS
    for name, (ret, params) in funcs.items():
        restype, argtypes = nccl._SIGNATURES[name]
        assert restype is _ctype(ret), name
        assert [_ctype(p) for p in params] == argtypes, name
        fn = getattr(nlib, name)
        assert fn.restype is restype and list(fn.argtypes) == argtypes, name
    assert defines["TRPL_NCCL_ID_BYTES"] == nccl.ID_BYTES
    assert defines["TRPL_ENCCL"] == nccl.ENCCL and defines["TRPL_ETIMEDOUT"] == nccl.ETIMEDOUT
    assert nlib.trpl_nccl_version() >= 21400        # non-blocking communicators


def test_return_code_contract(nlib):
    out = ctypes.c_void_p()
    i = ctypes.c_int()
    uid = ctypes.create_string_buffer(128)
    cases = [
        (nlib.trpl_nccl_unique_id(None), EINVAL),
        (nlib.trpl_nccl_comm_init(None, 1, 0, 0, 1000, ctypes.byref(out)), EINVAL),
        (nlib.trpl_nccl_comm_init(uid, 1, 0, 0, 1000, None), EINVAL),
        (nlib.trpl_nccl_comm_init(uid, 0, 0, 0, 1000, ctypes.byref(out)), EINVAL),
        (nlib.trpl_nccl_comm_init(uid, 2, -1, 0, 1000, ctypes.byref(out)), EINVAL),
        (nlib.trpl_nccl_comm_init(uid, 2, 2, 0, 1000, ctypes.byref(out)), EINVAL),
        (nlib.trpl_nccl_comm_init(uid, 1, 0, 0, 0, ctypes.byref(out)), EINVAL),
        (nlib.trpl_nccl_comm_init(uid, 1, 0, -1, 1000, ctypes.byref(out)), ENODEVICE),
        (nlib.trpl_nccl_comm_destroy(None), 0),
        (nlib.trpl_nccl_rank_info(None, ctypes.byref(i), ctypes.byref(i), ctypes.byref(i)), EINVAL),
        (nlib.trpl_allgather_rows(None, P, 1, 10, 10, 10, P, None), EINVAL),
        (nlib.trpl_logsumexp_nccl(None, P, 1, 10, 10, P, None), EINVAL),
        (nlib.trpl_allreduce_sum_nccl(None, P, 10, None), EINVAL),
        (nlib.trpl_posterior_weights_dev(None, 1, 10, 10, P, P, -1, None), EINVAL),
        (nlib.trpl_posterior_weights_dev(P, 1, 10, 10, None, P, -1, None), EINVAL),
        (nlib.trpl_posterior_weights_dev(P, 0, 10, 10, P, P, -1, None), EINVAL),
        (nlib.trpl_posterior_weights_dev(P, 1, 9, 10, P, P, -1, None), EINVAL),
        (nlib.trpl_posterior_weights_dev(P, 1, 10, 10, P, P, -1, None), ENODEVICE),
    ]
    assert [rc for rc, _ in cases] == [want for _, want in cases]
    assert out.value is None


def _needed(path):
    out = subprocess.run(["readelf", "-d", path], check=True, capture_output=True, text=True).stdout
    return re.findall(r"\(NEEDED\).*\[(.+)\]", out)


def test_only_the_companion_links_nccl(nlib):
    from bayesian_inference_trpl_b200 import _lib, nccl
    assert not [n for n in _needed(_lib.LIB_PATH) if "nccl" in n]
    assert "libnccl.so.2" in _needed(nccl.LIB_PATH)


def test_no_batched_memcpy_in_sources():
    """Copies go through cudaMemcpyAsync; the batched copy calls are kept out of every source and script."""
    pattern = re.compile(r"\bcu(da)?Memcpy(3D)?Batch" + "Async")
    sources = [os.path.join(ROOT, f) for f in os.listdir(ROOT) if os.path.isfile(os.path.join(ROOT, f))]
    for top in ("bayesian_inference_trpl_b200", "include", "oracle", "baseline", "tools", "profiles", "tests"):
        for d, dirs, files in os.walk(os.path.join(ROOT, top)):
            dirs[:] = [x for x in dirs if x not in ("__pycache__", "_ref")]    # _ref: unmodified reference copies
            sources += [os.path.join(d, f) for f in files]
    hits = []
    for path in sources:
        f = os.path.basename(path)
        if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cc", ".cpp", ".sh")) or f == "Makefile":
            with open(path, errors="replace") as fh:
                if pattern.search(fh.read()):
                    hits.append(os.path.relpath(path, ROOT))
    assert hits == []


# ---------------------------------------------------------------------------------------------------------
# one process, one rank
# ---------------------------------------------------------------------------------------------------------
def _spread_table(S=1001, seed=5):
    """[4, S]: values spread over +-700 with NaN and -inf entries; an all -inf row; a narrow row; a row whose
    first 400 columns hold no finite entry."""
    rng = np.random.default_rng(seed)
    t = rng.uniform(-700.0, 700.0, (4, S))
    t[0, rng.choice(S, 40, replace=False)] = np.nan
    t[0, rng.choice(S, 40, replace=False)] = -np.inf
    t[1] = -np.inf
    t[2] = rng.normal(-30.0, 2.0, S)
    t[3, :400] = np.where(np.arange(400) % 2 == 0, np.nan, -np.inf)
    return t


def _lse_ref(t):
    from scipy.special import logsumexp
    return np.array([logsumexp(r[np.isfinite(r)]) if np.isfinite(r).any() else -np.inf for r in t])


@pytest.fixture(scope="module")
def comm(nlib):
    torch = pytest.importorskip("torch")
    from bayesian_inference_trpl_b200 import nccl
    with nccl.Communicator(nccl.unique_id(), 0, 1, torch.cuda.current_device()) as c:
        yield c


def _exchange_all(c, x, lnp):
    """gather, lse, normalize and all-reduce of one rank, in that order on the current stream."""
    return (c.gather_rows(x, x.shape[-1]), c.global_logsumexp(x), c.normalize(lnp),
            c.allreduce_sum_(x.clone()))


@pytest.mark.gpu
def test_one_rank_exchange(comm):
    import torch
    from bayesian_inference_trpl_b200 import engine
    t = _spread_table()
    x = torch.from_numpy(t).cuda()
    np.testing.assert_array_equal(comm.gather_rows(x, t.shape[1]).cpu().numpy(), t)
    np.testing.assert_array_equal(comm.gather_rows(x[2], t.shape[1]).cpu().numpy(), t[2])
    lse = comm.global_logsumexp(x)
    assert lse.shape == (4,) and lse.is_cuda
    got = lse.cpu().numpy()
    ref = _lse_ref(t)
    assert got[1] == -np.inf
    np.testing.assert_allclose(got, ref, rtol=1e-13)
    one = comm.global_logsumexp(x[0])
    assert one.dim() == 0
    np.testing.assert_allclose(float(one), got[0], rtol=1e-14)       # block partials are added atomically
    np.testing.assert_array_equal(comm.allreduce_sum_(x.clone()).cpu().numpy(), t)
    # device-resident lse: the same bits as trpl_posterior_weights given that lse as a double; -inf row -> 0
    w = comm.posterior_weights(x, lse)
    for r in (0, 2, 3):
        assert torch.equal(w[r], engine.posterior_weights(x[r].contiguous(), float(lse[r])))
    assert (w[1] == 0).all()
    np.testing.assert_allclose(w.sum(dim=1).cpu().numpy()[[0, 2, 3]], 1.0, rtol=0, atol=1e-12)


@pytest.mark.gpu
def test_normalize_equals_the_engine_path(comm):
    import torch
    from bayesian_inference_trpl_b200 import TrplError, engine, posterior
    # 256 samples: one block per reduction, so the log-evidence is reproducible to the bit
    lnp = torch.from_numpy(np.random.default_rng(2).normal(-40.0, 5.0, 256)).cuda()
    lnp[7] = float("nan")
    w = comm.normalize(lnp)
    lse = float(posterior.log_evidence(lnp))
    assert torch.equal(w, engine.posterior_weights(lnp, lse))
    assert abs(float(w.sum()) - 1.0) <= 1e-12 and float(w[7]) == 0.0
    with pytest.raises(TrplError):
        comm.gather_rows(lnp[:10], 11)                    # one rank must hold all 11 columns


@pytest.mark.gpu
def test_shard_rule_is_checked(comm, nlib):
    import torch
    x = torch.zeros(2, 6, dtype=torch.float64, device="cuda")
    out = torch.empty(2, 7, dtype=torch.float64, device="cuda")
    lse = torch.empty(2, dtype=torch.float64, device="cuda")
    h = comm._handle()
    assert nlib.trpl_allgather_rows(h, x.data_ptr(), 2, 6, 6, 7, out.data_ptr(), None) == EINVAL
    assert nlib.trpl_allgather_rows(h, x.data_ptr(), 0, 6, 6, 6, out.data_ptr(), None) == EINVAL
    assert nlib.trpl_allgather_rows(h, x.data_ptr(), 2, 5, 6, 6, out.data_ptr(), None) == EINVAL
    assert nlib.trpl_logsumexp_nccl(h, x.data_ptr(), 0, 6, 6, lse.data_ptr(), None) == EINVAL
    rank, nranks, dev = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    assert nlib.trpl_nccl_rank_info(h, ctypes.byref(rank), ctypes.byref(nranks), ctypes.byref(dev)) == 0
    assert (rank.value, nranks.value, dev.value) == (0, 1, comm.device.index)


@pytest.mark.gpu
def test_stream_ordered_on_a_side_stream(comm):
    """Enqueued on a non-default stream right after the torch kernel that writes the input, with no host
    synchronisation in between, the results are those of the default stream (the log-sum-exp reductions
    add block partials atomically, so their last bits may differ between two calls)."""
    import torch
    t = _spread_table(S=200_003, seed=9)
    src = torch.from_numpy(t).cuda()
    lnp_src = torch.from_numpy(t[2].copy()).cuda()
    torch.cuda.synchronize()
    want = [v.cpu() for v in _exchange_all(comm, src, lnp_src)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        x = torch.empty_like(src)
        lnp = torch.empty_like(lnp_src)
        x.copy_(src)
        lnp.copy_(lnp_src)
        got = _exchange_all(comm, x, lnp)
    side.synchronize()
    exact = (True, False, False, True)
    for g, w, e in zip(got, want, exact):
        if e:
            np.testing.assert_array_equal(g.cpu().numpy(), w.numpy())
        else:
            np.testing.assert_allclose(g.cpu().numpy(), w.numpy(), rtol=1e-13, atol=0)


def _write_inputs(tmp_path, T=240):
    """Excitation and observation files of test_gpu_round2's product-path tests (small shape)."""
    import bayesian_inference_trpl_b200 as trpl
    from oracle import oracle
    from helpers import TRUTH, UC, example_data
    L, Time = 128, 0.025 * T
    exc_path = str(tmp_path / "exc.csv")
    with open(exc_path, "w") as fh:
        for row in example_data()["power_exc"]:
            fh.write(",".join("%.8E" % v for v in row) + ",\n")
    inis = trpl.bayes_io.get_initpoints(exc_path, {"select_obs_sets": None})
    simPar = [2000.0, Time, L, T, 1, (0,), 7, 10000]
    pls = [oracle.solve((TRUTH * UC)[None, :12], simPar, inis[c], solver="thomas")["pl"][0] for c in range(3)]
    obs_path = str(tmp_path / "obs.csv")
    trpl.bayes_io.write_observations(obs_path, [np.linspace(0, Time, T + 1)] * 3, pls)
    return exc_path, obs_path


def _config(sampler, T=240):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    cfg = parallel_bayes_gpu.default_config()
    cfg.update(Length=2000.0, Time=0.025 * T, T=T)
    cfg["ic_flags"]["time_cutoff"] = 0.025 * T
    cfg["sim_flags"].update(num_points=9, sampler=sampler)
    cfg["gpu_info"]["sims_per_gpu"] = 4
    return cfg


def _outputs(out):
    b = os.path.basename(out)
    return [np.load(os.path.join(out, "%s_BAYRAN_%s.npy" % (b, k))) for k in "PXW"]


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["numpy", "philox"])
def test_run_with_a_communicator_writes_the_default_files(comm, tmp_path, sampler):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    exc, obs = _write_inputs(tmp_path)
    outs = {}
    for name, ex in (("DEF", None), ("CAB", comm)):
        outs[name] = str(tmp_path / name)
        parallel_bayes_gpu.run(exc, [obs], [outs[name]], cfg=_config(sampler), seed=7, posterior=True, exchange=ex)
    for a, b in zip(_outputs(outs["DEF"]), _outputs(outs["CAB"])):
        np.testing.assert_array_equal(a, b)
    if sampler == "numpy":                                 # the command line, with a communicator of its own
        out = str(tmp_path / "CLI")
        parallel_bayes_gpu.main([exc, out, obs, "--num-points", "9", "--length", "2000", "--time-steps", "240",
                                 "--final-time", str(0.025 * 240), "--sims-per-gpu", "4", "--posterior",
                                 "--exchange", "cabi"])
        cli = _outputs(out)
        ref = str(tmp_path / "CLIREF")
        parallel_bayes_gpu.main([exc, ref, obs, "--num-points", "9", "--length", "2000", "--time-steps", "240",
                                 "--final-time", str(0.025 * 240), "--sims-per-gpu", "4", "--posterior"])
        for a, b in zip(_outputs(ref), cli):
            np.testing.assert_array_equal(a, b)


# ---------------------------------------------------------------------------------------------------------
# several processes, one GPU each
# ---------------------------------------------------------------------------------------------------------
def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


multi_gpu = pytest.mark.skipif(_ngpu() < 2, reason="needs at least 2 GPUs")
CHILD_TIMEOUT = 180.0

_CHILD_EXCHANGE = r"""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.environ["TRPL_ROOT"])
sys.path.insert(0, os.path.join(os.environ["TRPL_ROOT"], "tests"))
from bayesian_inference_trpl_b200 import distributed, engine, nccl
from test_nccl_exchange import _multi_inputs
rank, n, tmp = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), os.environ["TRPL_TMP"]
torch.cuda.set_device(rank)
t, X = _multi_inputs()
S = t.shape[1]
lo, hi = distributed.shard_bounds(S, rank, n)
with nccl.Communicator.from_file(os.path.join(tmp, "nccl.id"), rank, n, rank, timeout=120) as comm:
    assert not torch.distributed.is_initialized()
    local = torch.from_numpy(t[:, lo:hi].copy()).cuda()
    g = comm.gather_rows(local, S)
    lse = comm.global_logsumexp(local)
    w = comm.normalize(local)
    wsum = comm.allreduce_sum_(w.sum(dim=1))
    h = comm.allreduce_sum_(engine.weighted_hist(torch.from_numpy(X[lo:hi].copy()).cuda(), 0, w[0].contiguous(),
                                                 0.0, 1.0, 16))
    res = dict(gather=g.cpu().numpy(), lse=lse.cpu().numpy(), w=w.cpu().numpy(), wsum=wsum.cpu().numpy(),
               hist=h.cpu().numpy(), version=nccl.version())
    assert not torch.distributed.is_initialized()
np.savez(os.path.join(tmp, "rank%d.npz" % rank), **res)
"""

_CHILD_RUN = r"""
import os, sys
import torch
sys.path.insert(0, os.environ["TRPL_ROOT"])
sys.path.insert(0, os.path.join(os.environ["TRPL_ROOT"], "tests"))
from bayesian_inference_trpl_b200 import parallel_bayes_gpu
from test_nccl_exchange import _config
tmp = os.environ["TRPL_TMP"]
parallel_bayes_gpu.run(os.path.join(tmp, "exc.csv"), [os.path.join(tmp, "obs.csv")], [os.path.join(tmp, "MULTI")],
                       cfg=_config("numpy"), seed=7, posterior=True, exchange="cabi",
                       nccl_id_file=os.path.join(tmp, "run.id"))
assert not torch.distributed.is_initialized()
"""


def _multi_inputs():
    """Table [E=2, S=1001] (uneven shards on every world size up to 4) and a sample column in [0, 1]."""
    t = _spread_table(S=1001, seed=11)[[0, 3]]
    X = np.random.default_rng(12).uniform(0.0, 1.0, (1001, 13))
    return np.ascontiguousarray(t), X


def _spawn(script, n, tmp_path):
    """Run `script` in n child processes (RANK/WORLD_SIZE/LOCAL_RANK like torchrun); every child is killed and
    reaped before this returns."""
    procs, logs = [], []
    flags = ["-s"] if sys.flags.no_user_site else []
    try:
        for r in range(n):
            env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(n), LOCAL_RANK=str(r), TRPL_ROOT=ROOT,
                       TRPL_TMP=str(tmp_path))
            log = open(tmp_path / ("rank%d.log" % r), "w")
            logs.append(log)
            procs.append(subprocess.Popen([sys.executable] + flags + ["-c", script], env=env, cwd=ROOT,
                                          stdout=log, stderr=subprocess.STDOUT))
        deadline = time.monotonic() + CHILD_TIMEOUT
        for p in procs:
            try:
                p.wait(timeout=max(0.1, deadline - time.monotonic()))
            except subprocess.TimeoutExpired:
                break
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
            p.wait()
        for log in logs:
            log.close()
    failed = [(r, p.returncode) for r, p in enumerate(procs) if p.returncode != 0]
    if failed:
        tails = "\n".join("--- rank %d (exit %s):\n%s" % (r, rc, (tmp_path / ("rank%d.log" % r)).read_text()[-3000:])
                          for r, rc in failed)
        pytest.fail("child processes failed or timed out after %.0f s:\n%s" % (CHILD_TIMEOUT, tails))


@pytest.mark.gpu
@multi_gpu
def test_ranks_in_separate_processes_agree_with_one_process(nlib, tmp_path):
    import torch
    from bayesian_inference_trpl_b200 import engine, nccl
    n = min(_ngpu(), 4)
    _spawn(_CHILD_EXCHANGE, n, tmp_path)
    t, X = _multi_inputs()
    res = [np.load(tmp_path / ("rank%d.npz" % r)) for r in range(n)]
    print("NCCL %d, %d GPUs, %d ranks" % (int(res[0]["version"]), _ngpu(), n))
    lse_ref = _lse_ref(t)
    w_ref = np.where(np.isnan(t), 0.0, np.exp(t - lse_ref[:, None]))
    w_all = np.concatenate([r["w"] for r in res], axis=1)
    hist_ref = engine.weighted_hist(torch.from_numpy(X).cuda(), 0, torch.from_numpy(w_all[0].copy()).cuda(),
                                    0.0, 1.0, 16).cpu().numpy()
    for r in res:
        np.testing.assert_array_equal(r["gather"], t)
        np.testing.assert_allclose(r["lse"], lse_ref, rtol=1e-13)
        np.testing.assert_allclose(r["wsum"], 1.0, rtol=0, atol=1e-12)
        np.testing.assert_allclose(r["hist"], hist_ref, rtol=1e-12, atol=1e-300)
        assert int(r["version"]) == int(res[0]["version"])
    np.testing.assert_allclose(w_all, w_ref, rtol=1e-12, atol=0)
    assert nccl.version() >= 21400


@pytest.mark.gpu
@multi_gpu
def test_two_rank_run_over_the_c_abi_matches_one_rank(tmp_path):
    from bayesian_inference_trpl_b200 import parallel_bayes_gpu
    exc, obs = _write_inputs(tmp_path)
    one = str(tmp_path / "ONE")
    parallel_bayes_gpu.run(exc, [obs], [one], cfg=_config("numpy"), seed=7, posterior=True)
    _spawn(_CHILD_RUN, 2, tmp_path)
    P1, X1, W1 = _outputs(one)
    P2, X2, W2 = _outputs(str(tmp_path / "MULTI"))
    np.testing.assert_array_equal(P2, P1)
    np.testing.assert_array_equal(X2, X1)
    np.testing.assert_allclose(W2, W1, rtol=1e-12, atol=0)
