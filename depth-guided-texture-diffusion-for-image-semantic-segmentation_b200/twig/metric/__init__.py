"""Evaluation metrics of the reference's test path on the GPU (SURVEY.md 8f-4): mirrors of twig/metric/MAE.py,
Smeasure.py, Fmeasure.py, Emeasure.py and WeightedFmeasure.py (same class names, `process` / `compute_metrics`
protocol and result keys), and `SODEvaluator`, the whole table of pysodmetrics' `get_results()` in one evaluator."""
from .sod import (MAE, Emeasure, Fmeasure, Smeasure, SODEvaluator, WeightedFmeasure, sod_metrics,  # noqa: F401
                  sod_metrics_full, weighted_fmeasure)
