"""ctypes binding of libtrpl_b200.so (C ABI declared in include/trpl_b200.h).

The shared library is built in-tree by `build()` (nvcc, sm_100a only).  There is no CPU
fallback: if the library is missing or no B200 is visible, calls raise.
"""
import ctypes
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.environ.get("TRPL_LIB", os.path.join(_PKG, "libtrpl_b200.so"))   # TRPL_LIB: A/B-test builds
SRC = os.path.join(_PKG, "csrc", "trpl_kernels.cu")
INCLUDE = os.path.join(_ROOT, "include")

MAX_CURVES = 8
MAX_EXP = 4
OK, EINVAL, EUNSUPPORTED, ECUDA, ENODEVICE = 0, -1, -2, -3, -4
F64, F32 = 0, 1
F_INIT_GRID_UNITS, F_LOG_PL, F_SELF_NORMALIZE, F_EMULATE_F32 = 1, 2, 4, 8

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


class TrplError(RuntimeError):
    pass


class Obs(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int32), ("hi_max", ctypes.c_int32),
                ("d_hi", ctypes.c_void_p), ("d_whi", ctypes.c_void_p),
                ("d_wlo", ctypes.c_void_p), ("d_val", ctypes.c_void_p)]


class Curve(ctypes.Structure):
    _fields_ = [("d_init", ctypes.c_void_p), ("length", ctypes.c_double),
                ("obs", Obs * MAX_EXP)]


_vp, _int, _i64, _u64, _dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double

# name -> (restype, argtypes) of every export, in the order of include/trpl_b200.h
_SIGNATURES = {
    "trpl_version": (_int, []),
    "trpl_error_string": (ctypes.c_char_p, [_int]),
    "trpl_last_cuda_error": (ctypes.c_char_p, []),
    "trpl_resident_sims": (_int, [_int, _int]),
    "trpl_solve_pl": (_int, [_vp, _i64, _i64, _vp, _dbl, _dbl, _int, _int, _int, _int, _int, _int, _int,
                             _vp, _int, _i64, _vp, _vp, _int, _vp]),
    "trpl_solve_loglik": (_int, [_vp, _i64, _i64, _int, ctypes.POINTER(Curve), _int, _int, _dbl, _int,
                                 _int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _int, _vp]),
    "trpl_log10_clamp": (_int, [_vp, _int, _i64, _dbl, _int, _vp]),
    "trpl_lnp_accumulate": (_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _int, _vp]),
    "trpl_obs_prepare": (_int, [_vp, _int, _dbl, _int, _vp, _vp, _vp]),
    "trpl_lse_partial": (_int, [_vp, _i64, _vp, _int, _vp]),
    "trpl_random_grid": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _int, _int, _u64, _u64, _int, _vp]),
    "trpl_posterior_weights": (_int, [_vp, _i64, _dbl, _vp, _int, _vp]),
    "trpl_weighted_hist": (_int, [_vp, _i64, _i64, _int, _int, _vp, _dbl, _dbl, _int, _dbl, _dbl, _int, _vp,
                                  _int, _vp]),
    "trpl_weighted_moments": (_int, [_vp, _i64, _i64, _int, _vp, _vp, _int, _vp]),
    "trpl_selftest_rcp": (_int, [_vp, _vp, _i64, _int, _vp]),
    "trpl_bench_dfma": (_int, [_int, _int, ctypes.POINTER(_dbl), ctypes.POINTER(_dbl)]),
}
EXPORTS = list(_SIGNATURES)


def build(force=False, verbose=False):
    """Compile csrc/trpl_kernels.cu into libtrpl_b200.so for sm_100a (cross-compiles without a GPU)."""
    csrc = os.path.dirname(SRC)
    deps = [os.path.join(INCLUDE, "trpl_b200.h")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                     if f.endswith((".cu", ".cuh"))]
    if (not force and os.path.exists(LIB_PATH)
            and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(d) for d in deps)):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    cmd = [nvcc] + NVCC_FLAGS + ["-I", INCLUDE, "-o", LIB_PATH, SRC]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(cmd, env=env)
    return LIB_PATH


_lib = None


def lib():
    """Load the library (never builds implicitly on a GPU box: the .so ships with the snapshot)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TrplError("libtrpl_b200.so is not built: run `python -c 'import __graft_entry__ as g; "
                        "g.build()'` (needs nvcc). There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = L
    return L


def check(rc, what):
    if rc < 0:
        L = lib()
        msg = L.trpl_error_string(rc).decode()
        if rc == ECUDA:
            msg += " [" + L.trpl_last_cuda_error().decode() + "]"
        raise TrplError("%s failed: %s (code %d)" % (what, msg, rc))
    return rc
