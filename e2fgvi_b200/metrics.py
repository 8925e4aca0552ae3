"""Per-frame PSNR / SSIM of the reference's ``evaluate.py`` (``core/metrics.py:20-53``) on the GPU.

``psnr_ssim`` scores a batch of frames in one call of the ``e2f_psnr_ssim`` kernel (``csrc/metrics.cu``): fp64
throughout, deterministic, and a frame's result does not depend on the rest of the batch.  ``calc_psnr_and_ssim``
is a drop-in for the reference function of the same name.

There is no CPU path: CPU tensors raise.
"""
import numpy as np
import torch

from . import _lib
from .ops import _need_cuda, _stream


def psnr_ssim(ref_u8, test, win_size=65, data_range=255.0):
    """PSNR and SSIM of ``test`` against ``ref_u8`` per frame -> ``(psnr, ssim)``, fp64 CUDA tensors of shape (N,).

    ``ref_u8`` is (N,H,W,3) or (H,W,3) uint8 (the original frames); ``test`` has the same shape, fp32 (the canvas) or
    uint8 (converted to fp32, which is exact).  SSIM is scikit-image 0.16's ``compare_ssim(ref, test, data_range,
    multichannel=True, win_size)``; PSNR is ``20 log10(data_range / sqrt(mse))``, ``inf`` for equal frames."""
    if ref_u8.dtype != torch.uint8:
        raise TypeError(f"ref_u8 must be uint8, got {ref_u8.dtype}")
    if test.dtype == torch.uint8:
        test = test.float()
    if test.dtype != torch.float32:
        raise TypeError(f"test must be float32 or uint8, got {test.dtype}")
    if ref_u8.shape != test.shape or ref_u8.dim() not in (3, 4) or ref_u8.shape[-1] != 3:
        raise ValueError(f"expected two (N,H,W,3) or (H,W,3) arrays of one shape, got {tuple(ref_u8.shape)} and "
                         f"{tuple(test.shape)}")
    if ref_u8.device != test.device:
        raise ValueError(f"ref_u8 is on {ref_u8.device}, test on {test.device}")
    ref_u8, test = ref_u8.contiguous(), test.contiguous()
    n = ref_u8.shape[0] if ref_u8.dim() == 4 else 1
    h, w = ref_u8.shape[-3:-1]
    if win_size < 3 or win_size % 2 == 0:
        raise ValueError("Window size must be odd.")                      # skimage 0.16 compare_ssim's checks
    if win_size > min(h, w):
        raise ValueError("win_size exceeds image extent.  If the input is a multichannel (color) image, set "
                         "multichannel=True.")
    _need_cuda(ref_u8, test)
    lib = _lib.load()
    dev = ref_u8.device
    psnr = torch.empty(n, dtype=torch.float64, device=dev)
    ssim = torch.empty(n, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        if n == 0:
            return psnr, ssim
        ws = torch.empty(max(lib.e2f_psnr_ssim_workspace_bytes(n, h, w, win_size) // 8, 1), dtype=torch.float64,
                         device=dev)
        st = lib.e2f_psnr_ssim(ref_u8.data_ptr(), test.data_ptr(), psnr.data_ptr(), ssim.data_ptr(), n, h, w, win_size,
                               float(data_range), ws.data_ptr(), _stream())
        _lib.check(st, "e2f_psnr_ssim")
    return psnr, ssim


def calc_psnr_and_ssim(img1, img2):
    """``core/metrics.py:39``: numpy HWC images in [0, 255] (``img1`` the original, ``img2`` the result) -> two floats,
    computed on the current CUDA device.  ``img1`` must hold integers in [0, 255]; ``img2`` must be exact in fp32 (a
    uint8 image or an evaluation canvas)."""
    a = np.asarray(img1)
    b = np.asarray(img2)
    a8 = a.astype(np.uint8)
    if not np.array_equal(a8, a):
        raise ValueError("img1 must hold integers in [0, 255]")
    b32 = b.astype(np.float32)
    if not np.array_equal(b32, b):
        raise ValueError("img2 is not exact in float32")
    dev = torch.device("cuda", torch.cuda.current_device())
    p, s = psnr_ssim(torch.from_numpy(np.ascontiguousarray(a8)).to(dev), torch.from_numpy(np.ascontiguousarray(b32)).to(dev))
    return float(p[0]), float(s[0])
