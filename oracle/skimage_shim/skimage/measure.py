"""``skimage.measure.compare_ssim`` (0.16.2) for the call in core/metrics.py:47-51, backed by the fp64 restatement in
``oracle/restate_metrics.py`` (loaded by path: the repository root must stay off ``sys.path`` next to the
reference, whose ``model`` package the repository's ``model`` alias would shadow)."""
import importlib.util
import os

_spec = importlib.util.spec_from_file_location(
    "_restate_metrics", os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", "restate_metrics.py"))
_rm = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(_rm)


def compare_ssim(X, Y, win_size=None, gradient=False, data_range=None, multichannel=False, gaussian_weights=False,
                 full=False, **kwargs):
    if gradient or full or gaussian_weights or kwargs or win_size is None or data_range is None:
        raise NotImplementedError("only compare_ssim(X, Y, win_size=..., data_range=..., multichannel=...) is restated")
    if X.shape != Y.shape:
        raise ValueError("Input images must have the same dimensions.")
    if multichannel:
        return _rm.ssim(X, Y, win_size=win_size, data_range=data_range)
    return _rm.ssim_channel(X, Y, win_size=win_size, data_range=data_range)
