"""Evaluation metrics of the reference's test path on the GPU (SURVEY.md 8f-4): mirrors of twig/metric/MAE.py,
Smeasure.py, Fmeasure.py, Emeasure.py and WeightedFmeasure.py (same class names, `process` / `compute_metrics`
protocol and result keys)."""
from .sod import MAE, Emeasure, Fmeasure, Smeasure, WeightedFmeasure, sod_metrics, weighted_fmeasure  # noqa: F401
