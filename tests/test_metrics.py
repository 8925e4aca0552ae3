"""Frame metrics of evaluate.py: the fp64 oracle against a direct-window computation (CPU), the C ABI's argument
checks (CPU), and on the GPU the ``e2f_psnr_ssim`` kernel against the oracle, its exactness and determinism
properties, and the values the unmodified evaluate.py computed on the goldens' canvases."""
import os

import numpy as np
import pytest
import torch

from oracle import restate_metrics as RM

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _pair(kind, h, w, seed, n=None):
    """(original uint8, test) of one kind: random uint8 pairs, a quarter-integer canvas, or arbitrary fp32 in
    [0, 255]."""
    rng = np.random.default_rng(seed)
    shape = (h, w, 3) if n is None else (n, h, w, 3)
    a = rng.integers(0, 256, shape, dtype=np.uint8)
    if kind == "uint8":
        b = rng.integers(0, 256, shape, dtype=np.uint8).astype(np.float32)
    elif kind == "quarter":
        b = np.clip(a + rng.integers(-40, 41, shape) / 4.0, 0, 255).astype(np.float32)
    else:
        b = np.clip(a + rng.normal(0, 9, shape), 0, 255).astype(np.float32)
    return a, b


def _direct_ssim(a, b, win):
    return float(np.mean([RM.ssim_channel_direct(a[..., c], b[..., c], win) for c in range(3)]))


CPU_CASES = [(65, 65, 65), (65, 200, 65), (97, 131, 65), (65, 65, 7), (65, 200, 7), (97, 131, 7)]


@pytest.mark.parametrize("h,w,win", CPU_CASES)
@pytest.mark.parametrize("kind", ["uint8", "quarter", "fp32"])
def test_oracle_equals_direct_windows(h, w, win, kind):
    a, b = _pair(kind, h, w, h * 1000 + w + win)
    assert abs(RM.ssim(a, b, win_size=win) - _direct_ssim(a, b, win)) <= 1e-12
    mse = ((a.astype(np.float64) - b.astype(np.float64)) ** 2).sum() / a.size
    assert abs(RM.psnr(a, b) - 20 * np.log10(255 / np.sqrt(mse))) <= 1e-12


def test_oracle_identical_and_bad_windows():
    a, _ = _pair("uint8", 70, 80, 1)
    assert RM.psnr(a, a) == float("inf") and RM.ssim(a, a) == 1.0
    with pytest.raises(ValueError):
        RM.ssim(a, a, win_size=8)
    with pytest.raises(ValueError):
        RM.ssim(a, a, win_size=71)


def test_argument_errors_without_gpu(lib):
    """e2f_psnr_ssim validates before any CUDA call."""
    ok = (16, 16, 16, 16, 2, 240, 432, 65, 255.0, 16, None)
    call = lambda **kw: lib.e2f_psnr_ssim(*[kw.get(k, v) for k, v in zip(
        ("ref", "test", "psnr", "ssim", "n", "h", "w", "win", "dr", "ws", "stream"), ok)])
    assert call(ref=None) == -1 and b"null" in lib.e2f_last_error()
    assert call(ws=None) == -1
    assert call(win=64) == -1 and b"odd" in lib.e2f_last_error()
    assert call(win=1) == -1
    assert call(h=64) == -1 and b"exceeds" in lib.e2f_last_error()
    assert call(n=0) == -1 and call(h=0) == -1 and call(w=-1) == -1
    assert call(dr=0.0) == -1
    assert call(test=18) == -3 and call(psnr=12) == -3 and call(ws=4) == -3
    assert call(h=600, w=600, win=257) == -2
    assert lib.e2f_psnr_ssim_workspace_bytes(2, 240, 432, 64) == 0
    assert lib.e2f_psnr_ssim_workspace_bytes(2, 240, 432, 65) > 0
    assert lib.e2f_psnr_ssim_workspace_bytes(4, 240, 432, 65) == 2 * lib.e2f_psnr_ssim_workspace_bytes(2, 240, 432, 65)


def test_wrapper_checks_without_gpu():
    from e2fgvi_b200 import metrics
    a = torch.zeros(2, 40, 50, 3, dtype=torch.uint8)
    with pytest.raises(ValueError):
        metrics.psnr_ssim(a, a.float(), win_size=6)
    with pytest.raises(ValueError):
        metrics.psnr_ssim(a, a.float(), win_size=41)
    with pytest.raises(ValueError):
        metrics.psnr_ssim(a, a[:1].float(), win_size=7)
    with pytest.raises(TypeError):
        metrics.psnr_ssim(a.float(), a.float(), win_size=7)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.psnr_ssim(a, a.float(), win_size=7)


# ------------------------------------------------------------------------------------------------------------- GPU
def _oracle(a, b, win=65):
    a = a.reshape((-1,) + a.shape[-3:])
    b = b.reshape((-1,) + b.shape[-3:])
    return (np.array([RM.psnr(x, y) for x, y in zip(a, b)]), np.array([RM.ssim(x, y, win) for x, y in zip(a, b)]))


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,win", CPU_CASES + [(240, 432, 65), (240, 432, 7)])
@pytest.mark.parametrize("kind", ["uint8", "quarter", "fp32"])
def test_kernel_matches_oracle(cuda, h, w, win, kind):
    from e2fgvi_b200 import metrics
    a, b = _pair(kind, h, w, h + w + win, n=3)
    p, s = metrics.psnr_ssim(torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda), win_size=win)
    wp, ws = _oracle(a, b, win)
    assert p.dtype == torch.float64 and p.shape == (3,)
    assert np.abs(p.cpu().numpy() - wp).max() <= 1e-9
    assert np.abs(s.cpu().numpy() - ws).max() <= 1e-9


@pytest.mark.gpu
def test_kernel_batch_of_64_deterministic_and_batch_independent(cuda):
    from e2fgvi_b200 import metrics, ops
    a, b = _pair("quarter", 240, 432, 7, n=64)
    b[5] = a[5]                                                  # identical frame
    ad, bd = torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)
    n0 = ops.launch_count()
    p, s = metrics.psnr_ssim(ad, bd)
    assert ops.launch_count() - n0 == 2
    wp, ws = _oracle(a, b)
    p, s = p.cpu().numpy(), s.cpu().numpy()
    assert p[5] == float("inf") and s[5] == 1.0
    fin = np.isfinite(wp)
    assert np.abs(p[fin] - wp[fin]).max() <= 1e-9 and np.abs(s - ws).max() <= 1e-9
    p2, s2 = metrics.psnr_ssim(ad, bd)
    assert np.array_equal(p2.cpu().numpy(), p) and np.array_equal(s2.cpu().numpy(), s)
    for k in (0, 5, 31, 63):
        pk, sk = metrics.psnr_ssim(ad[k], bd[k])
        assert pk.item() == p[k] and sk.item() == s[k]
    pk, sk = metrics.psnr_ssim(ad[10:20], bd[10:20])
    assert np.array_equal(pk.cpu().numpy(), p[10:20]) and np.array_equal(sk.cpu().numpy(), s[10:20])


@pytest.mark.gpu
def test_uint8_and_fp32_inputs_agree_bitwise(cuda):
    from e2fgvi_b200 import metrics
    a, b = _pair("uint8", 100, 150, 3, n=4)
    ad, bd = torch.from_numpy(a).to(cuda), torch.from_numpy(b.astype(np.uint8)).to(cuda)
    p1, s1 = metrics.psnr_ssim(ad, bd, win_size=7)
    p2, s2 = metrics.psnr_ssim(ad, bd.float(), win_size=7)
    assert torch.equal(p1, p2) and torch.equal(s1, s2)
    pi, si = metrics.psnr_ssim(ad, ad)
    assert torch.all(torch.isinf(pi)) and torch.all(si == 1.0)


@pytest.mark.gpu
def test_calc_psnr_and_ssim_drop_in(cuda):
    from e2fgvi_b200 import metrics
    a, b = _pair("quarter", 240, 432, 9)
    p, s = metrics.calc_psnr_and_ssim(a, b)
    wp, ws = RM.calc_psnr_and_ssim(a, b)
    assert isinstance(p, float) and abs(p - wp) <= 1e-9 and abs(s - ws) <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["eval_e2fgvi", "eval_hq"])
def test_kernel_reproduces_evaluate_py_values(cuda, name, tmp_path):
    """On the canvas the unmodified evaluate.py scored, the kernel gives the PSNR / SSIM it computed."""
    from e2fgvi_b200 import metrics
    from test_evaluate import golden_case
    frames, masks, canvas, g = golden_case(name, tmp_path)
    p, s = metrics.psnr_ssim(torch.from_numpy(frames).to(cuda), torch.from_numpy(canvas).to(cuda))
    assert np.abs(p.cpu().numpy() - g["psnr"]).max() <= 1e-9
    assert np.abs(s.cpu().numpy() - g["ssim"]).max() <= 1e-9
