"""Parity against the UNMODIFIED reference run NATIVELY on a B200 (numba-CUDA `pvSimPCR.pvSim`,
`probs.py`, `bayeslib.bayes`), SURVEY 8(c) "exact oracle, GPU box".

Two sources for the reference side:
  * live: `baseline/_ref/` (a git-ignored copy of the reference's source, when present) is imported
    and run on the same GPU, same inputs, inside the test;
  * committed fixtures `tests/golden/ref_b200_*.npz`: outputs of that same code on a B200, written by
    `tools/ref_on_b200.py` (16 samples x 3 curves of the full T=80000 PL curves sub-sampled in time;
    the 256-sample likelihood table of the reference's `bayeslib.bayes`).

PL criterion everywhere: |PL - PL_ref| <= 1e-6*|PL_ref| + K*floor, floor = 2^12*eps*B*n0*p0*Length
(tests/helpers.pl_noise_floor): PL = rate*(sum N*P - L*N0*P0) cancels, so once the excess carriers are
gone the value is rounding noise of the equilibrium term (pvSimPCR.py:278-281).  Measured on 384 prior
samples x 80001 steps (profiles/r02_reference_parity.txt): two IEEE-division FP64 evaluations of the
reference algorithm (oracle Thomas vs oracle PCR = the reference's kernels) differ by up to 0.9 floor
there, this engine (reciprocal-multiply divisions, 1.5 ulp instead of 0.5) by up to 4.4 floors; K = 8.
The floor term only matters once PL has fallen ~12 decades below PL(0).
"""
import os
import sys

import numpy as np
import pytest

from helpers import (TRUTH, UC, golden, pl_noise_floor, power_scan_excitations, prior_samples,
                     route_a_case)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_FLOOR = 8.0


def _pl_excess(pl, ref, floor, rtol=1e-6):
    """err / (rtol*|ref| + K*floor): <= 1 everywhere means parity."""
    return np.abs(pl - ref) / (rtol * np.abs(ref) + K_FLOOR * floor[:, None])


def _golden_case():
    g = golden("ref_b200_pvsim.npz")
    sp = g["simPar"]
    simPar = [float(sp[0]), float(sp[1]), int(sp[2]), int(sp[3]), 1, (0,), int(sp[5]), int(sp[6])]
    return g, simPar


# ------------------------------------------------------------------------------------------------
# CPU: the oracle against the native reference at the full shape (80 001 steps: BDF5 steady
# state, Auger on) -- the long-run pin the <=24-step simulator goldens cannot give
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [0, 2])
def test_oracle_matches_native_reference_full_shape(curve):
    from oracle import oracle
    g, simPar = _golden_case()
    rows = [0, 3, 5, 7, 9, 14]
    X = g["X"][rows]
    ref = g["pl_ref_c%d" % curve][rows]
    pl = oracle.solve(X[:, :12], simPar, g["inis"][curve], solver="thomas")["pl"][:, g["t_idx"]]
    floor = pl_noise_floor(X[:, :12], simPar[0], simPar[1], simPar[2], simPar[3])
    assert _pl_excess(pl, ref, floor).max() <= 1.0
    # ... and in fact to 1e-9 over all 80 001 steps (Thomas vs the reference's PCR, both FP64)
    assert _pl_excess(pl, ref, floor, rtol=1e-9).max() <= 1.0


def test_oracle_pipeline_matches_native_reference_bayes():
    """oracle.loglik(emulate_f32) vs the likelihood table the reference's own bayeslib.bayes wrote on a
    B200 (f32 PL buffer, log10f, scipy griddata interpolation, probs.prob)."""
    from oracle import oracle
    g = golden("ref_b200_bayes.npz")
    inis = power_scan_excitations()
    case = route_a_case(inis, int(g["S"]), int(g["T"]))
    case["e_data"][0][1].extend(g["v_obs%d" % c] for c in range(3))
    n = 24
    P = oracle.loglik(g["X"][:n], case["simPar"], inis, case["e_data"], emulate_f32=True, solver="thomas")
    np.testing.assert_allclose(P[0], g["P_ref"][0][:n], rtol=5e-6)


# ------------------------------------------------------------------------------------------------
# GPU: this engine against the committed B200 outputs of the reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_pvsim_matches_native_reference_golden_full_shape():
    import bayesian_inference_trpl_b200 as trpl
    g, simPar = _golden_case()
    X = g["X"]
    floor = pl_noise_floor(X[:, :12], simPar[0], simPar[1], simPar[2], simPar[3])
    for c in range(3):
        pl = np.empty((len(X), simPar[3] + 1))
        st = np.zeros(len(X), dtype=np.int32)
        trpl.pvSim(pl, None, None, None, X[:, :12], simPar, g["inis"][c], (128,), 0, 1, init_mode="points",
                   status_out=st)
        assert (st == 0).all()
        ref = g["pl_ref_c%d" % c]
        ex = _pl_excess(pl[:, g["t_idx"]], ref, floor)
        assert ex.max() <= 1.0, "curve %d: worst excess %.3g at %s" % (c, ex.max(), np.unravel_index(ex.argmax(), ex.shape))
        tight = _pl_excess(pl[:, g["t_idx"]], ref, floor, rtol=1e-9)
        print("curve %d: worst excess at rtol 1e-6: %.3g, at 1e-9: %.3g" % (c, ex.max(), tight.max()))
        assert (tight <= 1.0).mean() >= 0.99


@pytest.mark.gpu
def test_bayes_matches_native_reference_golden():
    """The package's own bayeslib.bayes (fused + float32 emulation, and the staged float32 pipeline)
    against the table the reference wrote on a B200."""
    import bayesian_inference_trpl_b200 as trpl
    g = golden("ref_b200_bayes.npz")
    inis = power_scan_excitations()
    case = route_a_case(inis, int(g["S"]), int(g["T"]))
    case["e_data"][0][1].extend(g["v_obs%d" % c] for c in range(3))
    for fused in (True, False):
        info = dict(case["info"], fused=fused, emulate_f32=True, sims_per_gpu=256)
        np.random.seed(42)
        N, P, X = trpl.bayeslib.bayes(trpl.pvSim, np.array([0]), None, case["lo"], case["hi"], case["do_log"],
                                      inis, list(case["simPar"]), case["e_data"], dict(case["flags"]), info)
        np.testing.assert_array_equal(X, g["X"])
        np.testing.assert_allclose(P, g["P_ref"], rtol=3e-5 if fused else 1e-9)


# ------------------------------------------------------------------------------------------------
# GPU, live: the reference itself on this GPU, when its source is in baseline/_ref
# ------------------------------------------------------------------------------------------------
def _live_reference():
    """(baseline.ref_runner, None) when the reference's source is in baseline/_ref and numba can run
    it on the GPU, else (None, the reason it cannot)."""
    sys.path.insert(0, ROOT)
    from baseline import ref_runner as rr
    if not rr.available():
        return None, "baseline/_ref (copy of the reference's source) is not present"
    try:
        from numba import cuda
        if not cuda.is_available():
            return None, "numba sees no CUDA device"
    except Exception as e:                                  # pragma: no cover
        return None, "numba.cuda unusable: %r" % (e,)
    return rr, None


def _check_pl_and_lnl(pl, ref, X, simPar, what):
    """PL criterion, then the likelihood of every sample whose curve stays clear of the cancellation
    floor, evaluated the same way on both sides (f64 log10, residual against the reference curve of
    the truth sample, row 0)."""
    floor = pl_noise_floor(X[:, :12], simPar[0], simPar[1], simPar[2], simPar[3])
    ex = _pl_excess(pl, ref, floor)
    assert ex.max() <= 1.0, "%s: worst excess %.3g" % (what, ex.max())
    clean = (np.abs(ref) > 1e6 * floor[:, None]).all(axis=1)
    assert clean.mean() > 0.5
    lr, lm = np.log10(ref[clean]), np.log10(pl[clean])
    tgt = np.log10(ref[0])
    l_ref = -((lr - tgt) ** 2).sum(axis=1)
    l_my = -((lm - tgt) ** 2).sum(axis=1)
    np.testing.assert_allclose(l_my[1:], l_ref[1:], rtol=1e-6)


@pytest.mark.gpu
def test_pvsim_matches_reference_numba_kernels_live():
    """pvSimPCR.pvSim (numba-CUDA, unmodified, float64 PL buffer) vs trpl.pvSim.  Live: the same 384
    prior samples, highest-power curve at the full T=80000, the two others over the first 8000 steps.
    Without the reference's source: its stored B200 output (16 prior samples, all 3 curves at the full
    T=80000, 578 time points; tests/golden/ref_b200_pvsim.npz)."""
    import bayesian_inference_trpl_b200 as trpl
    rr, _ = _live_reference()
    if rr is None:
        g, simPar = _golden_case()
        X = g["X"]
        for c in range(3):
            pl = np.empty((len(X), simPar[3] + 1))
            st = np.zeros(len(X), dtype=np.int32)
            trpl.pvSim(pl, None, None, None, X[:, :12], simPar, g["inis"][c], (128,), 0, 1, init_mode="points",
                       status_out=st)
            assert (st == 0).all()
            _check_pl_and_lnl(pl[:, g["t_idx"]], g["pl_ref_c%d" % c], X, simPar, "stored curve %d" % c)
        return
    inis = power_scan_excitations()
    S = 384
    X = prior_samples(S, seed=77)
    X[0] = TRUTH * UC
    for c, T in ((2, 80000), (0, 8000), (1, 8000)):
        simPar = [2000.0, 0.025 * T, 128, T, 1, (0,), 7, 10000]
        ref, _ = rr.ref_pvsim(X, simPar, inis[c])
        pl = np.empty_like(ref)
        st = np.zeros(S, dtype=np.int32)
        trpl.pvSim(pl, None, None, None, X[:, :12], simPar, inis[c], (128,), 0, 1, init_mode="points", status_out=st)
        assert (st == 0).all() and np.isfinite(ref).all()
        _check_pl_and_lnl(pl, ref, X, simPar, "curve %d" % c)


@pytest.mark.gpu
def test_reference_bayeslib_drives_the_dropins_live():
    """INTEGRATION.md route A: the reference's own, unmodified bayeslib.bayes with
    sys.modules["probs"] = trpl.probs and model = trpl.pvSim reproduces the likelihood table of the
    all-reference run (its numba solver, fastlog and prob kernels) on the same GPU.  What it checks is
    that unmodified source driving the drop-ins, so it needs that source in baseline/_ref."""
    import bayesian_inference_trpl_b200 as trpl
    from oracle import oracle
    rr, why = _live_reference()
    if rr is None:
        pytest.skip(why)
    inis = power_scan_excitations()
    T = 2000
    case = route_a_case(inis, 96, T, truth_pl=lambda c: oracle.solve(
        (TRUTH * UC)[None, :12], [2000.0, 0.025 * T, 128, T, 1, (0,), 7, 10000], inis[c], solver="thomas")["pl"][0])
    args = (case["lo"], case["hi"], case["do_log"], inis, case["simPar"], case["e_data"], case["flags"], case["info"])
    N1, P1, X1 = rr.ref_bayes("reference", *args)
    N2, P2, X2 = rr.ref_bayes("dropin", *args)
    np.testing.assert_array_equal(X1, X2)
    assert np.isfinite(P1).all()
    np.testing.assert_allclose(P2, P1, rtol=1e-9)
