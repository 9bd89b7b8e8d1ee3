"""pyascore_b200 -- B200-native PTM-localisation scoring behind pyAscore's `PyAscore` API.

Only the scoring hot path lives here (DESIGN.md).  The CUDA library is loaded on first use and
there is no CPU fallback: constructing a scorer without the built .so or without a GPU raises.
"""
from .ascore import PyAscore
from .batch import MultiScorer, Scorer, format_results, pin_batch, pinned_empty, score_typed
from .ptm_scoring import (PyBinnedSpectra, PyBinomialDist, PyFragmentGraph, PyLogMath, PyModifiedPeptide,
                          PyPowerSetSum)
from .parsing import IdentificationParser, MassCorrector, SpectraParser

__all__ = ["PyAscore", "Scorer", "MultiScorer", "format_results", "pin_batch", "pinned_empty", "score_typed", "PyBinnedSpectra", "PyBinomialDist",
           "PyFragmentGraph", "PyLogMath", "PyModifiedPeptide", "PyPowerSetSum", "IdentificationParser",
           "MassCorrector", "SpectraParser"]
