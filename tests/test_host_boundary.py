"""The host boundary of libtrpl_b200.so: the ctypes binding agrees with include/trpl_b200.h, every
entry point returns its documented code for bad arguments (checked before any launch, so these run
without a GPU), and pinned staging buffers are private to each host thread."""
import ctypes
import os
import re
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "trpl_b200.h")

EINVAL, EUNSUPPORTED, ENODEVICE = -1, -2, -4
P = ctypes.c_void_p(16)          # placeholder device pointer: no case below dereferences it


@pytest.fixture(scope="module")
def lib():
    import bayesian_inference_trpl_b200 as trpl
    trpl.build()
    return trpl._lib.lib()


def _header():
    """{name: (return type, [parameter types])} and {TRPL_* define: value} of the C header."""
    src = re.sub(r"/\*.*?\*/", " ", open(HEADER).read(), flags=re.S)
    defines = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(TRPL_\w+)\s+(-?\d+)\b", src)}
    src = re.sub(r"typedef struct.*?\}\s*\w+\s*;", " ", src, flags=re.S)
    src = re.sub(r"#.*", " ", src)
    funcs = {}
    for m in re.finditer(r"([\w\s\*]+?)\b(trpl_\w+)\s*\(([^)]*)\)\s*;", src):
        params = [" ".join(p.split()) for p in m.group(3).split(",")]
        params = [] if params == ["void"] else [re.sub(r"\s*\b\w+$", "", p) for p in params]
        funcs[m.group(2)] = (" ".join(m.group(1).split()), params)
    return funcs, defines


def _ctype(func, ctype):
    """ctypes class a C parameter or return type is bound as."""
    if ctype == "const char *":
        return ctypes.c_char_p
    if ctype.endswith("*"):
        if "trpl_curve" in ctype:
            return "POINTER(Curve)"
        if func == "trpl_bench_dfma":
            return ctypes.POINTER(ctypes.c_double)
        return ctypes.c_void_p
    return {"int": ctypes.c_int, "int32_t": ctypes.c_int, "int64_t": ctypes.c_int64,
            "uint64_t": ctypes.c_uint64, "double": ctypes.c_double}[ctype]


def test_binding_matches_header(lib):
    from bayesian_inference_trpl_b200 import _lib
    funcs, defines = _header()
    assert len(funcs) == 16
    assert set(funcs) == set(_lib.EXPORTS)
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name, (ret, params) in funcs.items():
        assert hasattr(raw, name), name
        fn = getattr(lib, name)
        assert fn.restype is _ctype(name, ret), name
        argtypes = list(fn.argtypes or [])
        assert len(argtypes) == len(params), name
        for i, (got, c) in enumerate(zip(argtypes, params)):
            want = _ctype(name, c)
            if want == "POINTER(Curve)":
                want = ctypes.POINTER(_lib.Curve)
            assert got is want, (name, i, c, got)
    mirrored = {k[len("TRPL_"):]: v for k, v in defines.items() if hasattr(_lib, k[len("TRPL_"):])}
    assert {"MAX_CURVES", "MAX_EXP", "F64", "F32", "F_INIT_GRID_UNITS", "F_LOG_PL", "F_SELF_NORMALIZE",
            "F_EMULATE_F32"} <= set(mirrored)
    for k, v in mirrored.items():
        assert getattr(_lib, k) == v, k
    assert lib.trpl_version() >= 100
    assert lib.trpl_error_string(-2).decode().startswith("unsupported")


def _solve_pl(lib, d_matpar=P, L=128, device=-1):
    return lib.trpl_solve_pl(d_matpar, 4, 12, P, 1000.0, 10.0, L, 100, 1, 7, 100, 5, 0, P, 0, 101,
                             None, None, device, None)


def _solve_loglik(lib, C=1, E=1, L=128, n=0):
    from bayesian_inference_trpl_b200 import _lib
    curves = (_lib.Curve * (_lib.MAX_CURVES + 1))()
    curves[0].d_init = 16
    curves[0].length = 1000.0
    curves[0].obs[0].n = n
    return lib.trpl_solve_loglik(P, 4, 13, 12, curves, C, E, 10.0, L, 100, 7, 100, 5, 0, P, P, None, None,
                                 -1, None)


def _random_grid(lib, d_x=P, ncol=13, device=-1):
    lo = np.zeros(17)
    hi = np.ones(17)
    dl = np.zeros(17, dtype=np.int32)
    return lib.trpl_random_grid(d_x, 4, 17, lo.ctypes.data, hi.ctypes.data, dl.ctypes.data, ncol, 0, 1, 0,
                                device, None)


def test_return_code_contract(lib):
    tf = ctypes.c_double()
    cases = [
        (lib.trpl_resident_sims(-1, 128), ENODEVICE),
        (lib.trpl_resident_sims(-1, 1), EINVAL),
        (lib.trpl_resident_sims(-1, 4096), EUNSUPPORTED),
        (_solve_pl(lib, d_matpar=None), EINVAL),
        (_solve_pl(lib), ENODEVICE),
        (_solve_pl(lib, L=4096), EUNSUPPORTED),
        (_solve_loglik(lib, C=9), EUNSUPPORTED),
        (_solve_loglik(lib, E=5), EUNSUPPORTED),
        (_solve_loglik(lib, L=1), EINVAL),
        # the observation sets are checked after the device is entered
        (_solve_loglik(lib, n=-1), ENODEVICE),
        (lib.trpl_weighted_hist(P, 10, 13, 0, 1, P, 0.0, 1.0, 100, 0.0, 1.0, 100, P, -1, None), EUNSUPPORTED),
        (lib.trpl_weighted_moments(P, 10, 16, 16, P, P, -1, None), EINVAL),
        (_random_grid(lib, ncol=17), EINVAL),
        (lib.trpl_lse_partial(None, 10, P, -1, None), EINVAL),
        (lib.trpl_lse_partial(P, 10, P, -1, None), ENODEVICE),
        (lib.trpl_selftest_rcp(P, P, 10, -1, None), ENODEVICE),
        (lib.trpl_bench_dfma(-1, 0, ctypes.byref(tf), None), EINVAL),
        (lib.trpl_bench_dfma(-1, 10, ctypes.byref(tf), None), ENODEVICE),
        (lib.trpl_log10_clamp(None, 0, 10, 1e-10, -1, None), EINVAL),
        (lib.trpl_log10_clamp(P, 0, 10, 1e-10, -1, None), ENODEVICE),
        (lib.trpl_lnp_accumulate(None, P, 4, 10, 10, P, P, -1, None), EINVAL),
        (lib.trpl_lnp_accumulate(P, P, 4, 10, 10, P, P, -1, None), ENODEVICE),
        (lib.trpl_posterior_weights(None, 10, 0.0, P, -1, None), EINVAL),
        (lib.trpl_posterior_weights(P, 10, 0.0, P, -1, None), ENODEVICE),
        (_random_grid(lib, d_x=None), EINVAL),
        (_random_grid(lib), ENODEVICE),
    ]
    assert [rc for rc, _ in cases] == [want for _, want in cases]


@pytest.mark.gpu
def test_pinned_staging_is_per_thread():
    import torch
    from bayesian_inference_trpl_b200 import engine
    mine = engine.pinned("X", (4, 13), torch.float64)
    assert engine.pinned("X", (4, 13), torch.float64) is mine
    theirs = []
    t = threading.Thread(target=lambda: theirs.append(engine.pinned("X", (4, 13), torch.float64)))
    t.start()
    t.join()
    assert theirs[0] is not mine
    assert theirs[0].shape == mine.shape and theirs[0].is_pinned()
