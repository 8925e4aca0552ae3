"""TEST INFRASTRUCTURE — generates tests/golden/*.pt by running the UNMODIFIED reference (through the mmcv
shim, torchvision standing in for mmcv's DCN) on deterministic synthetic weights and frames.

    python -m oracle.gen_golden            # only works where /root/reference exists (the build container)

Weights and inputs are NOT stored: they are regenerated bit-identically from (family, seed) by
``e2fgvi_b200.synth`` on any machine with the same torch; only the reference's outputs are committed.
"""
import importlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from e2fgvi_b200.synth import synth_frames, synth_state_dict  # noqa: E402
from oracle.reference_loader import import_reference, reference_generator  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# name -> (hq, H, W, T, l_t, family, weight seed, frame seed[, clips b, pixel subsample stride])
E2E_CASES = {
    "e2e_base_stress": (False, 240, 432, 8, 5, "stress", 0, 3),
    "e2e_base_default": (False, 240, 432, 8, 5, "default", 0, 3),
    "e2e_hq_tiny_stress": (True, 120, 216, 4, 3, "stress", 0, 5),
    "e2e_hq_small_stress": (True, 180, 324, 5, 3, "stress", 1, 6),
    # round 2: the shapes bench.py measures (BASELINE configs[2], [3] per-GPU share, [4]) and a mid-size 10+6 case.
    # Subsample strides are coprime with the 12-pixel token pitch and the 60x108-pixel attention window so that every
    # phase of the fold / window geometry is sampled.
    "e2e_base_b8_stress": (False, 240, 432, 8, 5, "stress", 0, 11, 8, 5),
    "e2e_hq720_stress": (True, 720, 1296, 8, 5, "stress", 2, 7, 1, 7),
    "e2e_hq360_t16_stress": (True, 360, 648, 16, 10, "stress", 3, 8, 1, 5),
    "e2e_hq1080_t16_stress": (True, 1080, 1944, 16, 10, "stress", 4, 9, 1, 11),
    # tests/test_oracle.py::test_oracle_vs_live_reference: a second HQ weight / frame draw, every 5th pixel
    "e2e_hq_tiny_s3_stress": (True, 120, 216, 4, 3, "stress", 3, 9, 1, 5),
}


def gen_e2e(only=None):
    import time
    for name, case in E2E_CASES.items():
        if only and name not in only:
            continue
        hq, H, W, T, lt, family, wseed, fseed = case[:8]
        b = case[8] if len(case) > 8 else 1
        t0 = time.time()
        ref = reference_generator(hq)
        mine = importlib.import_module("e2fgvi_b200.model." + ("e2fgvi_hq" if hq else "e2fgvi")).InpaintGenerator()
        sd = synth_state_dict(mine, family, wseed)
        ref.load_state_dict(sd, strict=True)
        x = synth_frames(b, T, H, W, seed=fseed)
        with torch.no_grad():
            pred, (ff, fb) = ref(x, lt)
        # full-size cases keep every 2nd pixel (exact fp32 values) + whole-tensor statistics to stay small in git
        sub = case[9] if len(case) > 9 else (2 if H * W > 100000 else 1)
        torch.save({"case": dict(hq=hq, H=H, W=W, T=T, l_t=lt, family=family, weight_seed=wseed, frame_seed=fseed, b=b),
                    "subsample": sub, "pred": pred[:, :, ::sub, ::sub].contiguous(),
                    "pred_sum": float(pred.double().sum()), "pred_abs_sum": float(pred.double().abs().sum()),
                    "flows_forward": ff.contiguous(), "flows_backward": fb.contiguous()},
                   os.path.join(OUT, name + ".pt"))
        print(name, tuple(pred.shape), float(pred.abs().max()), f"{time.time() - t0:.0f} s", flush=True)


def gen_ops():
    """Operator-level goldens from the reference's own modules / functions."""
    g = torch.Generator().manual_seed(1234)
    out = {}
    fc = import_reference("model.modules.flow_comp")
    x = torch.randn(2, 128, 12, 20, generator=g)
    flow = torch.randn(2, 12, 20, 2, generator=g) * 4.0
    out["flow_warp"] = {"x": x, "flow": flow,
                        "zeros": fc.flow_warp(x, flow, padding_mode="zeros"),
                        "border": fc.flow_warp(x, flow, padding_mode="border")}

    # SecondOrderDeformableAlignment of the reference (feat_prop.py:13-58), stress weights from the model dict
    fp = import_reference("model.modules.feat_prop")
    mine = importlib.import_module("e2fgvi_b200.model.e2fgvi").InpaintGenerator()
    sd = synth_state_dict(mine, "stress", 0)
    align = fp.SecondOrderDeformableAlignment(256, 128, 3, padding=1, deform_groups=16)
    pre = "feat_prop_module.deform_align.backward_."
    align.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=True)
    xa = torch.randn(1, 256, 10, 14, generator=g) * 0.5
    extra = torch.randn(1, 384, 10, 14, generator=g) * 0.5
    f1 = torch.randn(1, 2, 10, 14, generator=g) * 2.0
    f2 = torch.randn(1, 2, 10, 14, generator=g) * 2.0
    with torch.no_grad():
        out["deform_align"] = {"x": xa, "extra": extra, "flow_1": f1, "flow_2": f2,
                               "out": align(xa, extra, f1, f2)}

    # WindowAttention of the reference (tfocal_transformer.py:150-399) incl. qkv / proj, block-0 stress weights
    tf = import_reference("model.modules.tfocal_transformer")
    attn = tf.WindowAttention(512, (2, 4), (5, 9), (5, 9), 2, 4, True, "fc")
    pre = "transformer.0.attn."
    attn.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=True)
    xt = torch.randn(1, 2, 10, 18, 512, generator=g)
    pooled = torch.randn(1, 2, 2, 2, 512, generator=g)          # (B, nWh, nWw, T, C)
    with torch.no_grad():
        out["window_attention"] = {"x": xt, "pooled": pooled, "out": attn([xt, pooled], [None, None])}
    torch.save(out, os.path.join(OUT, "ops.pt"))
    print("ops", {k: tuple(v["out"].shape) if "out" in v else None for k, v in out.items()})


def gen_layout():
    """state_dict key / shape / dtype list of the reference generators (the checkpoint contract, SURVEY §8(b))."""
    import json
    layout = {}
    for hq in (False, True):
        sd = reference_generator(hq).state_dict()
        layout["e2fgvi_hq" if hq else "e2fgvi"] = [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()]
    with open(os.path.join(OUT, "state_dict_layout.json"), "w") as f:
        json.dump(layout, f, indent=0)
    print("layout", {k: len(v) for k, v in layout.items()})


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "--layout-only" in sys.argv:
        gen_layout()
        sys.exit(0)
    if "--e2e" in sys.argv:          # python -m oracle.gen_golden --e2e name [name ...]: only these end-to-end cases
        torch.set_num_threads(os.cpu_count())
        gen_e2e(set(sys.argv[sys.argv.index("--e2e") + 1:]))
        sys.exit(0)
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    gen_layout()
    gen_ops()
    gen_e2e()
