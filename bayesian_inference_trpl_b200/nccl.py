"""ctypes binding of libtrpl_b200_nccl.so (C ABI declared in include/trpl_b200_nccl.h): the end-of-run
exchange of a multi-GPU run over NCCL without torch.distributed, and `Communicator`, which offers it
with the contract of the `distributed` functions it replaces.

The library is a companion of libtrpl_b200.so, built in-tree by `build()` and linked with libnccl.so.2.
When torch is imported first, the dynamic loader reuses the libnccl.so.2 torch already loaded (it
matches by soname); `version()` reports the NCCL that actually runs.
"""
import ctypes
import os
import subprocess
import time

import numpy as np
import torch

from . import _lib, distributed

LIB_PATH = os.environ.get("TRPL_NCCL_LIB", os.path.join(_lib._PKG, "libtrpl_b200_nccl.so"))
SRC = os.path.join(_lib._PKG, "csrc", "trpl_nccl.cu")
HEADER = os.path.join(_lib.INCLUDE, "trpl_b200_nccl.h")

ID_BYTES = 128
OK, EINVAL, ECUDA, ENODEVICE, ENCCL, ETIMEDOUT = 0, -1, -3, -4, -5, -6
_MESSAGES = {EINVAL: "invalid argument", ECUDA: "CUDA runtime error", ENODEVICE: "no usable CUDA device",
             ENCCL: "NCCL error", ETIMEDOUT: "timed out waiting for the other ranks"}

_vp, _int, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64

# name -> (restype, argtypes) of every export, in the order of include/trpl_b200_nccl.h
_SIGNATURES = {
    "trpl_nccl_version": (_int, []),
    "trpl_nccl_last_error": (ctypes.c_char_p, []),
    "trpl_nccl_unique_id": (_int, [_vp]),
    "trpl_nccl_comm_init": (_int, [_vp, _int, _int, _int, _int, _vp]),
    "trpl_nccl_comm_destroy": (_int, [_vp]),
    "trpl_nccl_rank_info": (_int, [_vp, _vp, _vp, _vp]),
    "trpl_allgather_rows": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "trpl_logsumexp_nccl": (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "trpl_posterior_weights_dev": (_int, [_vp, _i64, _i64, _i64, _vp, _vp, _int, _vp]),
    "trpl_allreduce_sum_nccl": (_int, [_vp, _vp, _i64, _vp]),
}
EXPORTS = list(_SIGNATURES)


def build(force=False):
    """Compile csrc/trpl_nccl.cu into libtrpl_b200_nccl.so for sm_100a, linked with -lnccl."""
    csrc = os.path.dirname(SRC)
    deps = [HEADER, os.path.join(_lib.INCLUDE, "trpl_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cu", ".cuh"))]
    if (not force and os.path.exists(LIB_PATH)
            and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(d) for d in deps)):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc] + _lib.NVCC_FLAGS + ["-I", _lib.INCLUDE, "-o", LIB_PATH, SRC, "-lnccl"], env=env)
    return LIB_PATH


_nlib = None


def lib():
    """Load the library (never builds implicitly: the .so ships with the snapshot)."""
    global _nlib
    if _nlib is not None:
        return _nlib
    if not os.path.exists(LIB_PATH):
        raise _lib.TrplError("libtrpl_b200_nccl.so is not built: run `python -c 'import __graft_entry__ as g; "
                             "g.build()'` (needs nvcc and the NCCL headers).")
    L = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = restype, argtypes
    _nlib = L
    return L


def check(rc, what):
    if rc < 0:
        msg = _MESSAGES.get(rc, "unknown error")
        if rc in (ECUDA, ENCCL, ETIMEDOUT):
            msg += " [" + lib().trpl_nccl_last_error().decode() + "]"
        raise _lib.TrplError("%s failed: %s (code %d)" % (what, msg, rc))
    return rc


def version():
    """Runtime NCCL version code (e.g. 22703 for 2.27.3)."""
    return check(lib().trpl_nccl_version(), "trpl_nccl_version")


def unique_id():
    """A fresh communicator id (TRPL_NCCL_ID_BYTES bytes); made on rank 0 and handed to every rank."""
    buf = ctypes.create_string_buffer(ID_BYTES)
    check(lib().trpl_nccl_unique_id(buf), "trpl_nccl_unique_id")
    return buf.raw


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else None


def _rows(t):
    """A device tensor as [rows, n] with unit column stride (last dim = samples)."""
    t = t.contiguous()
    if t.dim() == 0:
        return t.reshape(1, 1)
    return t.reshape(int(np.prod(t.shape[:-1])), t.shape[-1])      # not -1: a rank may hold 0 columns


class Communicator:
    """One rank of an NCCL communicator on one GPU, used for the exchange at the end of a run.

    Collective methods must be called by every rank in the same order.  They are stream-ordered on the
    current torch stream of the communicator's device and return device tensors without synchronising the
    host.  Columns are sharded by `distributed.shard_bounds`."""

    def __init__(self, id_bytes, rank, nranks, device, timeout=120.0):
        if len(id_bytes) != ID_BYTES:
            raise ValueError("a communicator id has %d bytes" % ID_BYTES)
        self.rank, self.nranks = int(rank), int(nranks)
        self.device = torch.device("cuda", int(device))
        handle = ctypes.c_void_p()
        check(lib().trpl_nccl_comm_init(ctypes.c_char_p(bytes(id_bytes)), self.nranks, self.rank,
                                        self.device.index, int(timeout * 1000), ctypes.byref(handle)),
              "trpl_nccl_comm_init")
        self._comm = handle

    @classmethod
    def from_file(cls, path, rank, nranks, device, timeout=120.0):
        """Bootstrap through a file every rank can read: rank 0 writes a fresh id to `path` (atomically, via a
        temporary file and os.replace), the others wait up to `timeout` seconds for it.  `path` must not
        exist before the run (use one path per run)."""
        if int(rank) == 0:
            uid = unique_id()
            tmp = "%s.tmp%d" % (path, os.getpid())
            with open(tmp, "wb") as fh:
                fh.write(uid)
            os.replace(tmp, path)
        else:
            deadline = time.monotonic() + timeout
            while not os.path.exists(path):
                if time.monotonic() > deadline:
                    raise _lib.TrplError("no communicator id appeared at %s within %.0f s" % (path, timeout))
                time.sleep(0.01)
            with open(path, "rb") as fh:
                uid = fh.read()
        return cls(uid, rank, nranks, device, timeout=timeout)

    # -- lifetime ------------------------------------------------------------------------------------------
    def close(self):
        if self._comm is not None:
            comm, self._comm = self._comm, None
            check(lib().trpl_nccl_comm_destroy(comm), "trpl_nccl_comm_destroy")

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _handle(self):
        if self._comm is None:
            raise _lib.TrplError("the communicator is closed")
        return self._comm

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _local(self, t):
        if t.device != self.device or t.dtype != torch.float64:
            raise ValueError("expected a float64 tensor on %s" % self.device)
        return _rows(t)

    # -- exchange ------------------------------------------------------------------------------------------
    def rank_world(self):
        return self.rank, self.nranks

    def gather_rows(self, local, n_total):
        """All-gather contiguous shards (last dim = samples) into the full table on every rank
        (distributed.gather_rows)."""
        x = self._local(local)
        out = torch.empty(x.shape[0], int(n_total), dtype=torch.float64, device=self.device)
        check(lib().trpl_allgather_rows(self._handle(), _ptr(x), x.shape[0], x.shape[1], x.shape[1], int(n_total),
                                        _ptr(out), self._stream()), "trpl_allgather_rows")
        return out.reshape(local.shape[:-1] + (int(n_total),))

    def global_logsumexp(self, x):
        """log sum exp over all ranks' entries: a 0-d device tensor for a 1-D x, [rows] for a 2-D x (NaN
        skipped, -inf weighs 0, -inf when no rank has a finite entry)."""
        if x.dim() not in (1, 2):
            raise ValueError("x must be 1-D or 2-D")
        xr = self._local(x)
        lse = torch.empty(xr.shape[0], dtype=torch.float64, device=self.device)
        check(lib().trpl_logsumexp_nccl(self._handle(), _ptr(xr), xr.shape[0], xr.shape[1], xr.shape[1], _ptr(lse),
                                        self._stream()), "trpl_logsumexp_nccl")
        return lse[0] if x.dim() == 1 else lse

    def posterior_weights(self, lnP, lse):
        """exp(lnP - lse) on the device with lse a device tensor (one value per row), NaN -> 0."""
        x = self._local(lnP)
        lse = lse.reshape(-1).contiguous()
        if lse.numel() != x.shape[0]:
            raise ValueError("one lse per row of lnP is required")
        w = torch.empty_like(x)
        check(lib().trpl_posterior_weights_dev(_ptr(x), x.shape[0], x.shape[1], x.shape[1], _ptr(lse), _ptr(w),
                                               self.device.index, self._stream()), "trpl_posterior_weights_dev")
        return w.reshape(lnP.shape)

    def normalize(self, lnP):
        """Posterior weights of this rank's samples, summing to one over all ranks (posterior.normalize);
        the log-evidence never leaves the device."""
        return self.posterior_weights(lnP, self.global_logsumexp(lnP))

    def allreduce_sum_(self, t):
        """In-place sum over the ranks of a contiguous float64 device tensor."""
        if not t.is_contiguous():
            raise ValueError("allreduce_sum_ needs a contiguous tensor")
        self._local(t)
        check(lib().trpl_allreduce_sum_nccl(self._handle(), _ptr(t), t.numel(), self._stream()),
              "trpl_allreduce_sum_nccl")
        return t

    # -- the exchange points of parallel_bayes_gpu.run --------------------------------------------------
    def merge_block_cyclic(self, P_local):
        """distributed.merge_block_cyclic: sum the per-rank block-cyclic tables (device tensor result)."""
        if self.nranks == 1:
            return P_local
        t = torch.as_tensor(np.asarray(P_local), dtype=torch.float64).to(self.device)
        return self.allreduce_sum_(t)

    def posterior_weights_full(self, lnP):
        """Weights of a full table held by every rank: each rank normalises its shard against the global
        log-evidence and the shards are gathered back."""
        n = lnP.shape[-1]
        lo, hi = distributed.shard_bounds(n, self.rank, self.nranks)
        return self.gather_rows(self.normalize(lnP[..., lo:hi]), n)
