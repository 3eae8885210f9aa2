"""B200-native engine for the TRPL forward-model + likelihood hot path of
HagesLab/Bayesian-Inference-TRPL.  Python surface mirrors the reference:

    pvSim(...)                    <- pvSimPCR.pvSim        (pvSimPCR.py:309)
    fastlog(...), prob(...)       <- probs.fastlog / prob  (probs.py:78, :49)
    bayeslib.simulate / bayes     <- bayeslib.py:83, :207
    bayes_io.get_data / get_initpoints / export
    engine.solve_loglik           fused device-resident path (no reference counterpart)
"""
from . import _lib, bayes_io, bayes_validate, bayeslib, distributed, engine, probs, pvsim  # noqa: F401
from . import ensemble, parallel_bayes_gpu, posterior, tempering  # noqa: F401
from ._lib import TrplError, build  # noqa: F401
from .probs import fastlog, prob  # noqa: F401
from .pvsim import pvSim  # noqa: F401

__all__ = ["pvSim", "fastlog", "prob", "bayeslib", "bayes_io", "bayes_validate", "engine",
           "distributed", "build", "TrplError"]
