"""TEST INFRASTRUCTURE — numpy fp64 restatement of the frame metrics of the reference's ``evaluate.py``:
``core/metrics.py:20-36`` (``calculate_psnr``), ``:39-53`` (``calc_psnr_and_ssim``) and the scikit-image 0.16.2
``measure.compare_ssim`` it calls (``environment.yml:109``) with ``data_range=255, multichannel=True, win_size=65``.
Only tests/, ``oracle/gen_golden_eval.py`` and ``tools/eval_bench.py`` import it; the product path
(``e2fgvi_b200/metrics.py``) never does.

scikit-image is not installed here (and ``compare_ssim`` is gone from releases after 0.17), so this restatement is
pinned against a brute-force direct-window fp64 sum of the same formula on small images
(``tests/test_metrics.py``); agreement with skimage itself is by construction, not by a recorded run.
"""
import numpy as np
from scipy.ndimage import uniform_filter


def psnr(img1, img2, data_range=255.0):
    """``calculate_psnr`` (core/metrics.py:20-36) on float64 inputs; ``inf`` when the images are equal."""
    img1 = np.asarray(img1, np.float64)
    img2 = np.asarray(img2, np.float64)
    assert img1.shape == img2.shape
    mse = np.mean((img1 - img2) ** 2)
    if mse == 0:
        return float("inf")
    return float(20.0 * np.log10(data_range / np.sqrt(mse)))


def ssim_channel(x, y, win_size=65, data_range=255.0):
    """skimage 0.16 ``compare_ssim`` of two 2-D images (gaussian_weights=False, use_sample_covariance=True)."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    if win_size % 2 == 0 or win_size < 3:
        raise ValueError("Window size must be odd.")
    if any(s < win_size for s in x.shape):
        raise ValueError("win_size exceeds image extent.")
    np_ = win_size ** 2
    cov_norm = np_ / (np_ - 1)
    ux = uniform_filter(x, size=win_size)
    uy = uniform_filter(y, size=win_size)
    uxx = uniform_filter(x * x, size=win_size)
    uyy = uniform_filter(y * y, size=win_size)
    uxy = uniform_filter(x * y, size=win_size)
    vx = cov_norm * (uxx - ux * ux)
    vy = cov_norm * (uyy - uy * uy)
    vxy = cov_norm * (uxy - ux * uy)
    c1 = (0.01 * data_range) ** 2
    c2 = (0.03 * data_range) ** 2
    a1, a2, b1, b2 = 2 * ux * uy + c1, 2 * vxy + c2, ux ** 2 + uy ** 2 + c1, vx + vy + c2
    s = (a1 * a2) / (b1 * b2)
    pad = (win_size - 1) // 2
    return float(s[pad:s.shape[0] - pad, pad:s.shape[1] - pad].mean())


def ssim(img1, img2, win_size=65, data_range=255.0):
    """``compare_ssim(img1, img2, data_range, multichannel=True, win_size)``: the mean of the per-channel values."""
    img1 = np.asarray(img1)
    img2 = np.asarray(img2)
    assert img1.shape == img2.shape and img1.ndim == 3
    return float(np.mean([ssim_channel(img1[..., c], img2[..., c], win_size, data_range)
                          for c in range(img1.shape[-1])]))


def calc_psnr_and_ssim(img1, img2):
    """core/metrics.py:39-53: HWC images in [0, 255] -> (psnr, ssim)."""
    img1 = np.asarray(img1).astype(np.float64)
    img2 = np.asarray(img2).astype(np.float64)
    return psnr(img1, img2), ssim(img1, img2, win_size=65, data_range=255)


def ssim_channel_direct(x, y, win_size, data_range=255.0):
    """The same S, mean over the cropped outputs, with every window summed directly (no filter): the independent
    computation ``ssim_channel`` is checked against."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    h, w = x.shape
    pad = win_size // 2
    np_ = win_size ** 2
    cov_norm = np_ / (np_ - 1)
    c1 = (0.01 * data_range) ** 2
    c2 = (0.03 * data_range) ** 2
    vals = []
    for i in range(pad, h - pad):
        for j in range(pad, w - pad):
            wx = x[i - pad:i + pad + 1, j - pad:j + pad + 1]
            wy = y[i - pad:i + pad + 1, j - pad:j + pad + 1]
            ux, uy = wx.sum() / np_, wy.sum() / np_
            vx = cov_norm * ((wx * wx).sum() / np_ - ux * ux)
            vy = cov_norm * ((wy * wy).sum() / np_ - uy * uy)
            vxy = cov_norm * ((wx * wy).sum() / np_ - ux * uy)
            vals.append((2 * ux * uy + c1) * (2 * vxy + c2) / ((ux * ux + uy * uy + c1) * (vx + vy + c2)))
    return float(np.mean(vals))
