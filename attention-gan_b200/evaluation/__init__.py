"""Evaluation of trained DAMSM encoders: R-precision scores on the B200 kernels (see r_precision.py)."""
from .r_precision import DAMSMScorer, mismatched_candidates, r_precision  # noqa: F401
