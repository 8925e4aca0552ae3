"""Minimal stand-in for scikit-image 0.16.2 so the reference's core/metrics.py imports offline (test infrastructure):
only ``measure.compare_ssim`` as evaluate.py calls it, backed by ``oracle/restate_metrics.py``."""
