"""Device-level API of the B200 TRPL engine: torch tensors are the buffers, libtrpl_b200.so does
the work (kernels in csrc/trpl_kernels.cu).  Nothing in here computes on the CPU.

Shapes follow the reference: simPar = [Length, Time, L, T, plT, pT, tol, MAX]
(parallel_bayes_gpu.py:81), X [S,13] with mag_offset last (parallel_bayes_gpu.py:84),
e_data = [(t_list, logPL_list, unc_list)] per observation file (bayes_io.py:99-102).
"""
import ctypes
import threading
import time

import numpy as np
import torch

from . import _lib
from ._lib import (F32, F64, F_EMULATE_F32, F_INIT_GRID_UNITS, F_LOG_PL, F_SELF_NORMALIZE,
                   MAX_CURVES, MAX_EXP, TrplError, check)


def require_cuda(device=None):
    if not torch.cuda.is_available():
        raise TrplError("no CUDA device visible: the TRPL engine has no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
    return dev


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _row_stride(t):
    # a single-row view may carry any (even 0) stride on its first axis
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _call(name, dev, *args):
    """Run export `name` with `args` on `dev` and its current stream (every stream-ordered export takes
    those two last); raise on a negative return code."""
    return check(getattr(_lib.lib(), name)(*args, dev.index, _stream(dev)), name)


def host_wait(dev=None):
    """Block the calling host thread until everything queued on the current stream has finished, by
    polling an event.  The driver's blocking waits (cudaDeviceSynchronize / cudaStreamSynchronize /
    cudaEventSynchronize, i.e. torch.cuda.synchronize and tensor.cpu()) were measured to return up to
    0.7 s late after a multi-second kernel on the B200 boxes of this pool (tools/sync_latency.py,
    profiles/r02_sync_latency.txt); polling learns of completion within 0.1 ms."""
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(dev))
    while not ev.query():
        time.sleep(0)           # yield the GIL / the core to other host threads between polls


def to_device_f64(a, dev):
    """Host array -> contiguous float64 device tensor through pinned memory."""
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=torch.float64).contiguous()
    h = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
    if h.numel() > 0:
        h = h.pin_memory()
    return h.to(dev, non_blocking=True)


class ObservationSet:
    """One curve of one observation file, bracketed on the step grid and resident on the device."""

    def __init__(self, times, values, Time, T, dev):
        times = np.ascontiguousarray(times, dtype=np.float64)
        values = np.ascontiguousarray(values, dtype=np.float64)
        if times.shape != values.shape or times.ndim != 1:
            raise ValueError("observation times/values must be 1-D and of equal length")
        n = times.shape[0]
        hi = np.empty(n, dtype=np.int32)
        whi = np.empty(n)
        wlo = np.empty(n)
        rc = _lib.lib().trpl_obs_prepare(
            times.ctypes.data_as(ctypes.c_void_p), n, float(Time), int(T),
            hi.ctypes.data_as(ctypes.c_void_p), whi.ctypes.data_as(ctypes.c_void_p),
            wlo.ctypes.data_as(ctypes.c_void_p))
        if rc < 0:
            raise ValueError("observation times must be sorted and lie inside [0, Time]")
        self.n = n
        self.hi_max = int(rc)
        self.hi = torch.from_numpy(hi).to(dev)
        self.whi = torch.from_numpy(whi).to(dev)
        self.wlo = torch.from_numpy(wlo).to(dev)
        self.val = torch.from_numpy(values).to(dev)

    def fill(self, obs):
        obs.n = self.n
        obs.hi_max = self.hi_max
        obs.d_hi = self.hi.data_ptr()
        obs.d_whi = self.whi.data_ptr()
        obs.d_wlo = self.wlo.data_ptr()
        obs.d_val = self.val.data_ptr()


class Problem:
    """Everything that is shared by all samples of a run, resident on one device: the excitation
    curves (iniPar rows), their thicknesses and the prepared observation sets of every file."""

    def __init__(self, simPar, iniPar, e_data, device=None, init_mode="points"):
        self.dev = require_cuda(device)
        Length, Time, L, T, plT, pT, tol, MAX = simPar
        if int(plT) != 1:
            raise ValueError("the fused likelihood path samples PL on every step (plT = 1, what bayeslib's "
                             "[S, T+1] buffer requires, bayeslib.py:137); got plT = %r" % (plT,))
        self.Time, self.L, self.T, self.tol, self.MAX = float(Time), int(L), int(T), int(tol), int(MAX)
        iniPar = np.asarray(iniPar, dtype=np.float64)
        self.C = iniPar.shape[0]
        if isinstance(Length, (list, tuple, np.ndarray)):
            self.lengths = [float(x) for x in Length]
        else:
            self.lengths = [float(Length)] * self.C
        if len(self.lengths) != self.C:
            raise ValueError("one thickness per excitation curve is required")
        self.E = len(e_data)
        if init_mode != "points":
            raise ValueError("Problem takes point-wise excitation profiles")
        self.init = [to_device_f64(iniPar[c], self.dev) for c in range(self.C)]
        self.obs = [[ObservationSet(exp[0][c], exp[1][c], self.Time, self.T, self.dev)
                     for c in range(self.C)] for exp in e_data]
        # One fused launch covers up to MAX_CURVES curves x MAX_EXP observation files; larger
        # problems are tiled (curve tiles accumulate into the same lnL rows, file tiles fill
        # different rows -- at the price of re-running the forward model for every file tile).
        self.parts = []
        for e0 in range(0, self.E, MAX_EXP):
            e1 = min(self.E, e0 + MAX_EXP)
            for c0 in range(0, self.C, MAX_CURVES):
                c1 = min(self.C, c0 + MAX_CURVES)
                curves = (_lib.Curve * (c1 - c0))()
                for c in range(c0, c1):
                    curves[c - c0].d_init = self.init[c].data_ptr()
                    curves[c - c0].length = self.lengths[c]
                    for e in range(e0, e1):
                        self.obs[e][c].fill(curves[c - c0].obs[e - e0])
                self.parts.append((e0, e1, c0, c1, curves))

    def steps_per_sample(self):
        """Time steps actually integrated per sample (sum over curves, causal truncation included)."""
        return sum(max(self.obs[e][c].hi_max for e in range(self.E)) + 1 for c in range(self.C))


_PROBLEMS = {}          # digest -> Problem, insertion-ordered (small LRU)
_STAGING = threading.local()   # .bufs: (tag, shape, dtype) -> pinned host staging tensor of one host thread


def cached_problem(simPar, iniPar, e_data, device=None, keep=4):
    """Problem for these inputs, staged on the device once and reused while the CONTENT of
    (simPar, iniPar, e_data) is unchanged (bayeslib.simulate is called once per run in the reference, but a
    driver that calls it per batch should not re-bracket and re-upload 240 k observations every time)."""
    import hashlib
    dev = require_cuda(device)
    h = hashlib.blake2b(digest_size=16)
    Length = simPar[0]
    h.update(repr((dev.index, [float(v) for v in np.atleast_1d(Length)], float(simPar[1]), int(simPar[2]),
                   int(simPar[3]), int(simPar[4]), int(simPar[6]), int(simPar[7]), len(e_data))).encode())
    h.update(np.ascontiguousarray(iniPar, dtype=np.float64).tobytes())
    for exp in e_data:
        for c in range(len(exp[0])):
            h.update(np.ascontiguousarray(exp[0][c], dtype=np.float64).tobytes())
            h.update(np.ascontiguousarray(exp[1][c], dtype=np.float64).tobytes())
    key = h.digest()
    prob = _PROBLEMS.pop(key, None)
    if prob is None:
        prob = Problem(simPar, iniPar, e_data, device=dev.index)
    _PROBLEMS[key] = prob
    while len(_PROBLEMS) > keep:
        _PROBLEMS.pop(next(iter(_PROBLEMS)))
    return prob


def pinned(tag, shape, dtype):
    """Reusable pinned host staging buffer of the calling thread.  Each host thread has its own, so
    threads that run the same batch shape never write and read one buffer around async copies."""
    bufs = getattr(_STAGING, "bufs", None)
    if bufs is None:
        bufs = _STAGING.bufs = {}
    key = (tag, tuple(shape), dtype)
    t = bufs.get(key)
    if t is None:
        if len(bufs) > 16:
            bufs.clear()
        t = torch.empty(tuple(shape), dtype=dtype).pin_memory()
        bufs[key] = t
    return t


def solve_pl(matpar, init, length, time, L, T, plT=1, tol=7, max_iter=10000, out_dtype=torch.float64,
             init_grid_units=False, max_order=5, want_iters=True):
    """pvSimPCR.pvSim on device tensors: returns (pl [S, T//plT+1], status [S] i32, iters [S] i64)."""
    dev = matpar.device
    if dev.type != "cuda":
        raise TrplError("matpar must be a CUDA tensor")
    assert matpar.dtype == torch.float64 and matpar.dim() == 2 and matpar.stride(1) == 1
    S = matpar.shape[0]
    npl = T // plT + 1
    pl = torch.empty((S, npl), dtype=out_dtype, device=dev)
    status = torch.zeros(S, dtype=torch.int32, device=dev)
    iters = torch.zeros(S, dtype=torch.int64, device=dev) if want_iters else None
    flags = F_INIT_GRID_UNITS if init_grid_units else 0
    _call("trpl_solve_pl", dev,
          _ptr(matpar), S, _row_stride(matpar), _ptr(init), float(length), float(time), int(L), int(T),
          int(plT), int(tol), int(max_iter), int(max_order), flags, _ptr(pl),
          F32 if out_dtype == torch.float32 else F64, npl, _ptr(status), _ptr(iters))
    return pl, status, iters


def solve_loglik(X, problem, log_pl=True, self_normalize=False, emulate_f32=False, lnl=None,
                 max_order=5, want_iters=False):
    """Fused forward model + likelihood for every row of X (device tensor [S, >=13]).

    Returns (lnl [E,S] f64, status [S] i32, iters [C,S] i64 or None).  `lnl` (if given) is
    accumulated into, like the reference's P (probs.py:60)."""
    dev = problem.dev
    assert X.device == dev and X.dtype == torch.float64 and X.dim() == 2 and X.stride(1) == 1
    S = X.shape[0]
    C, E = problem.C, problem.E
    if lnl is None:
        lnl = torch.zeros((E, S), dtype=torch.float64, device=dev)
    assert lnl.shape == (E, S) and lnl.is_contiguous()
    status = torch.zeros(S, dtype=torch.int32, device=dev)
    iters = torch.zeros((C, S), dtype=torch.int64, device=dev) if want_iters else None
    flags = ((F_LOG_PL if log_pl else 0) | (F_SELF_NORMALIZE if self_normalize else 0)
             | (F_EMULATE_F32 if emulate_f32 else 0))
    mag_col = 12 if X.shape[1] > 12 else -1
    for e0, e1, c0, c1, curves in problem.parts:
        sse = torch.empty((e1 - e0, c1 - c0, S), dtype=torch.float64, device=dev)
        st = status if len(problem.parts) == 1 else torch.zeros(S, dtype=torch.int32, device=dev)
        _call("trpl_solve_loglik", dev,
              _ptr(X), S, _row_stride(X), mag_col, curves, c1 - c0, e1 - e0, problem.Time, problem.L,
              problem.T, problem.tol, problem.MAX, int(max_order), flags, _ptr(sse), _ptr(lnl[e0:e1]),
              _ptr(st), _ptr(iters[c0:c1]) if (iters is not None and e0 == 0) else None)
        if st is not status:
            status |= st
    return lnl, status, iters


def log10_clamp_(t, MIN):
    """probs.fastlog on a device tensor (in place)."""
    assert t.is_cuda and t.is_contiguous() and t.dtype in (torch.float32, torch.float64)
    _call("trpl_log10_clamp", t.device, _ptr(t), F32 if t.dtype == torch.float32 else F64, t.numel(), float(MIN))
    return t


def lnp_accumulate_(P, pl, values, mag):
    """probs.prob on device tensors: P[j] -= sum_i (pl[j,i] + mag[j] - values[i])^2 (in place)."""
    assert P.is_cuda and pl.dtype == torch.float64 and pl.stride(1) == 1
    _call("trpl_lnp_accumulate", P.device,
          _ptr(P), _ptr(pl), pl.shape[0], pl.shape[1], pl.stride(0), _ptr(values), _ptr(mag))
    return P


def lse_partial(x):
    """(max, sum exp(x - max)) over the finite entries of a device vector -> tensor [2]."""
    assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous()
    out = torch.empty(2, dtype=torch.float64, device=x.device)
    _call("trpl_lse_partial", x.device, _ptr(x), x.numel(), _ptr(out))
    return out


def resident_sims(L, device=None):
    dev = require_cuda(device)
    return check(_lib.lib().trpl_resident_sims(dev.index, int(L)), "trpl_resident_sims")


def bench_dfma(iters=20000, device=None):
    dev = require_cuda(device)
    tf, ms = ctypes.c_double(), ctypes.c_double()
    check(_lib.lib().trpl_bench_dfma(dev.index, int(iters), ctypes.byref(tf), ctypes.byref(ms)),
          "trpl_bench_dfma")
    return tf.value, ms.value


def random_grid_device(minX, maxX, do_log, num_points, seed, first_sample=0, override_flags=0,
                       device=None, out=None):
    """bayeslib.random_grid/make_grid on the device (trpl_random_grid): X [num_points, ncol] CUDA tensor.
    Counter-based, so rank r can generate rows [lo, hi) of the global draw with first_sample=lo."""
    dev = require_cuda(device)
    lo = np.ascontiguousarray(minX, dtype=np.float64)
    hi = np.ascontiguousarray(maxX, dtype=np.float64)
    dl = np.ascontiguousarray(do_log, dtype=np.int32)
    ncol = lo.shape[0]
    X = out if out is not None else torch.empty((num_points, ncol), dtype=torch.float64, device=dev)
    _call("trpl_random_grid", dev, _ptr(X), num_points, _row_stride(X),
          lo.ctypes.data_as(ctypes.c_void_p), hi.ctypes.data_as(ctypes.c_void_p),
          dl.ctypes.data_as(ctypes.c_void_p), ncol, int(override_flags), int(seed), int(first_sample))
    return X


def posterior_weights(lnp, lse):
    """w = exp(lnP - lse) on the device (NaN -> 0)."""
    assert lnp.is_cuda and lnp.dtype == torch.float64 and lnp.is_contiguous()
    w = torch.empty_like(lnp)
    _call("trpl_posterior_weights", lnp.device, _ptr(lnp), lnp.numel(), float(lse), _ptr(w))
    return w


def weighted_hist(X, colx, w, lox, hix, nbx, coly=-1, loy=0.0, hiy=1.0, nby=1, out=None):
    """Raw weighted histogram (numpy.histogram / histogram2d binning) of column colx (x coly) of X."""
    assert X.is_cuda and X.dtype == torch.float64 and X.stride(1) == 1
    shape = (nbx,) if coly < 0 else (nbx, nby)
    h = out if out is not None else torch.zeros(shape, dtype=torch.float64, device=X.device)
    _call("trpl_weighted_hist", X.device, _ptr(X), X.shape[0], _row_stride(X), int(colx), int(coly), _ptr(w),
          float(lox), float(hix), int(nbx), float(loy), float(hiy), int(nby), _ptr(h))
    return h


def weighted_moments(X, w, ncol=None, out=None):
    """Raw sums [sum w, sum w x_j, sum w x_j x_k] of the first ncol columns of X."""
    assert X.is_cuda and X.dtype == torch.float64 and X.stride(1) == 1
    ncol = X.shape[1] if ncol is None else ncol
    o = out if out is not None else torch.zeros(1 + ncol + ncol * ncol, dtype=torch.float64, device=X.device)
    _call("trpl_weighted_moments", X.device, _ptr(X), X.shape[0], _row_stride(X), int(ncol), _ptr(w), _ptr(o))
    return o
