"""CPU: the oracle restatement against the goldens produced by the real reference."""
import importlib
import os

import pytest
import torch

from e2fgvi_b200.synth import synth_frames, synth_state_dict
from oracle import restate

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _sd(hq, family, seed):
    m = importlib.import_module("e2fgvi_b200.model." + ("e2fgvi_hq" if hq else "e2fgvi")).InpaintGenerator()
    return synth_state_dict(m, family, seed)


def test_ops_goldens():
    g = torch.load(os.path.join(GOLDEN, "ops.pt"))
    fw = g["flow_warp"]
    for pad in ("zeros", "border"):
        # the reference normalises to [-1,1] and grid_sample denormalises (fp32 round trip): <= 1e-5 on O(4) data
        assert (restate.flow_warp(fw["x"], fw["flow"], padding_mode=pad) - fw[pad]).abs().max() < 1e-5
    sd = _sd(False, "stress", 0)
    da = g["deform_align"]
    got = restate.deform_align(sd, "feat_prop_module.deform_align.backward_", da["x"], da["extra"], da["flow_1"],
                               da["flow_2"])
    assert (got - da["out"]).abs().max() < 1e-5
    wa = g["window_attention"]
    from e2fgvi_b200.model.modules.tfocal_transformer import rolled_valid_indices, window_partition
    pre = "transformer.0.attn."
    qkv = torch.nn.functional.linear(wa["x"], sd[pre + "qkv.weight"], sd[pre + "qkv.bias"])
    qkvp = torch.nn.functional.linear(wa["pooled"].permute(0, 3, 1, 2, 4), sd[pre + "qkv.weight"], sd[pre + "qkv.bias"])
    att = restate.focal_window_attention(qkv, qkvp, 4, (5, 9), (2, 4), (5, 9), 128 ** -0.5,
                                         rolled_valid_indices((5, 9), (2, 4)))
    out = torch.nn.functional.linear(window_partition(att, (5, 9)), sd[pre + "proj.weight"], sd[pre + "proj.bias"])
    assert (out - wa["out"]).abs().max() < 1e-4


@pytest.mark.parametrize("name", ["e2e_hq_tiny_stress", "e2e_hq_small_stress", "e2e_base_stress"])
def test_e2e_goldens(name):
    g = torch.load(os.path.join(GOLDEN, name + ".pt"))
    c = g["case"]
    sd = _sd(c["hq"], c["family"], c["weight_seed"])
    x = synth_frames(1, c["T"], c["H"], c["W"], seed=c["frame_seed"])
    with torch.no_grad():
        pred, (ff, fb) = restate.inpaint_generator_forward(sd, x, c["l_t"])
    s = g["subsample"]
    assert (pred[:, :, ::s, ::s] - g["pred"]).abs().max() < 5e-5          # both fp32 CPU: rounding order only
    assert abs(float(pred.double().sum()) - g["pred_sum"]) < 1e-2 * max(1.0, abs(g["pred_sum"])) + 5.0
    assert (ff - g["flows_forward"]).abs().max() < 1e-3
    assert (fb - g["flows_backward"]).abs().max() < 1e-3


def test_explicit_dcn_matches_torchvision():
    tv = pytest.importorskip("torchvision.ops")
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 32, 9, 11, generator=g)
    off = torch.randn(2, 72, 9, 11, generator=g) * 3
    msk = torch.rand(2, 36, 9, 11, generator=g)
    w = torch.randn(8, 32, 3, 3, generator=g)
    b = torch.randn(8, generator=g)
    a = restate.modulated_deform_conv2d(x, off, msk, w, b, 1, 1, 1, 1, 4)
    t = tv.deform_conv2d(x, off, w, b, (1, 1), (1, 1), (1, 1), mask=msk)
    assert (a - t).abs().max() < 1e-5


def test_oracle_vs_live_reference():
    """The HQ oracle against what the reference network computed on a second weight / frame draw (stored by
    ``python -m oracle.gen_golden --e2e e2e_hq_tiny_s3_stress``: every 5th pixel, whole-tensor sums, full flows)."""
    g = torch.load(os.path.join(GOLDEN, "e2e_hq_tiny_s3_stress.pt"))
    sd = _sd(True, "stress", 3)
    x = synth_frames(1, 4, 120, 216, seed=9)
    with torch.no_grad():
        got, gf = restate.inpaint_generator_forward(sd, x, 3)
    s = g["subsample"]
    assert (got[:, :, ::s, ::s] - g["pred"]).abs().max() < 5e-5
    assert abs(float(got.double().sum()) - g["pred_sum"]) / got.numel() < 1e-6
    assert abs(float(got.double().abs().sum()) - g["pred_abs_sum"]) / got.numel() < 1e-6
    assert (g["flows_forward"] - gf[0]).abs().max() < 1e-3 and (g["flows_backward"] - gf[1]).abs().max() < 1e-3
