"""Deterministic synthetic weights and frames.

No released checkpoint or dataset is reachable offline, so parity and benchmarks run on random-init weights and
synthetic frames (BASELINE.json).  Every tensor is drawn on the CPU from a ``torch.Generator`` seeded by
(seed, key), so the same values are produced in this container (where the goldens are made from the real
reference) and on the GPU box.

Two weight families:
* ``"default"``  — the reference's construction-time family: N(0,0.02) convs/linears with zero bias
  (e2fgvi.py:29-68), zeroed last offset conv (feat_prop.py:32-33), uniform DCN weight, kaiming SPyNet.
  Activations shrink to ~1e-2 and offsets equal the flow, so this family alone is a weak parity test (SURVEY §7).
* ``"stress"``   — fan-in-scaled weights so activations stay O(1), non-zero biases, a live last offset conv
  (offsets = flow + up to +-10 px, masks spread over (0,1)), perturbed LayerNorm / pooling weights.
"""
import hashlib
import math

import torch

FAMILIES = ("default", "stress")


def _gen(seed, key):
    h = hashlib.sha256(f"{seed}:{key}".encode()).digest()
    g = torch.Generator(device="cpu")
    g.manual_seed(int.from_bytes(h[:8], "little") & 0x7FFFFFFFFFFFFFFF)
    return g


def _normal(shape, std, g, mean=0.0):
    return torch.empty(shape, dtype=torch.float32).normal_(mean, std, generator=g)


def _fan_in(shape):
    return int(math.prod(shape[1:])) if len(shape) > 1 else int(shape[0])


def synth_state_dict(model, family="default", seed=0):
    """Return a full ``state_dict`` (CPU, fp32 / int64) for ``model`` with deterministic synthetic values."""
    if family not in FAMILIES:
        raise ValueError(f"family must be one of {FAMILIES}")
    ref = model.state_dict()
    out = {}
    stress = family == "stress"
    for key in sorted(ref.keys()):
        t = ref[key]
        shape = tuple(t.shape)
        g = _gen(seed, key)
        leaf = key.rsplit(".", 1)[-1]
        if not t.is_floating_point():  # attn.valid_ind_rolled: structural, keep the constructed value
            out[key] = t.detach().cpu().clone()
            continue
        if key.startswith("update_spynet."):
            if leaf in ("mean", "std"):
                out[key] = t.detach().cpu().clone()
            elif leaf == "weight":  # kaiming-normal fan_out / relu, what mmcv's ConvModule does by default
                fan_out = shape[0] * shape[2] * shape[3]
                out[key] = _normal(shape, math.sqrt(2.0 / fan_out), g)
                if stress and ".basic_module.4.conv." in key:
                    out[key] *= 0.06  # keeps |flow| at a few pixels so warps sample inside the map
            else:
                out[key] = _normal(shape, 0.02, g) if stress else torch.zeros(shape)
            continue
        if ".norm1." in key or ".norm2." in key:
            if leaf == "weight":
                out[key] = 1.0 + (_normal(shape, 0.1, g) if stress else 0.0) * torch.ones(shape)
            else:
                out[key] = _normal(shape, 0.1, g) if stress else torch.zeros(shape)
            continue
        if key == "sc.bias":
            out[key] = _normal(shape, 0.1, g) if stress else torch.zeros(shape)
            continue
        if ".pool_layers." in key:
            if leaf == "weight":
                out[key] = (1.0 / shape[1] + _normal(shape, 0.01, g)) if stress else _normal(shape, 0.02, g)
            else:
                out[key] = _normal(shape, 0.05, g) if stress else torch.zeros(shape)
            continue
        is_dcn = ".deform_align." in key and ".conv_offset." not in key
        is_last_offset = ".conv_offset.6." in key
        if leaf == "weight":
            fan = _fan_in(shape)
            if is_dcn:
                bound = 1.0 / math.sqrt(fan)
                w = torch.empty(shape).uniform_(-bound, bound, generator=g)
                out[key] = w * (math.sqrt(3.0) if stress else 1.0)  # stress: unit-variance-preserving
            elif is_last_offset:
                out[key] = _normal(shape, 0.6 / math.sqrt(fan), g) if stress else torch.zeros(shape)
            elif stress:
                out[key] = _normal(shape, 1.0 / math.sqrt(fan), g)
            else:
                out[key] = _normal(shape, 0.02, g)
        elif leaf == "bias":
            if is_last_offset:
                out[key] = _normal(shape, 0.3, g) if stress else torch.zeros(shape)
            else:
                out[key] = _normal(shape, 0.05, g) if stress else torch.zeros(shape)
        else:
            raise KeyError(f"no synthetic rule for {key}")
    return out


def synth_frames(b, t, h, w, seed=0, holes=True):
    """``masked_frames`` (b,t,3,h,w) fp32 in [-1,1]: smooth moving texture + noise, with a zeroed rectangle per
    frame (what test.py:155 feeds the model: imgs*(1-mask))."""
    g = _gen(seed, f"frames:{b}:{t}:{h}:{w}")
    yy = torch.linspace(0, 1, h).view(1, 1, 1, h, 1)
    xx = torch.linspace(0, 1, w).view(1, 1, 1, 1, w)
    tt = torch.arange(t, dtype=torch.float32).view(1, t, 1, 1, 1)
    ph = torch.rand((b, 1, 3, 1, 1), generator=g) * 6.28
    base = 0.5 * torch.sin(6.28 * (2.0 * xx + 0.03 * tt) + ph) * torch.cos(6.28 * (1.5 * yy - 0.02 * tt))
    x = (base + 0.5 * (torch.rand((b, t, 3, h, w), generator=g) * 2 - 1)).clamp_(-1, 1)
    if holes:
        hh, ww = max(h // 4, 1), max(w // 4, 1)
        for bi in range(b):
            for ti in range(t):
                y0 = int(torch.randint(0, h - hh + 1, (1,), generator=g))
                x0 = int(torch.randint(0, w - ww + 1, (1,), generator=g))
                x[bi, ti, :, y0:y0 + hh, x0:x0 + ww] = 0.0
    return x.contiguous()


def synth_video(n, h, w, seed=0):
    """A synthetic RGB video and its hole masks for the video-level driver (test.py:125-141):
    ``frames`` (n,h,w,3) uint8 — drifting sinusoid texture + noise — and ``masks`` (n,h,w) uint8 in {0,1} — a
    rectangle that moves across the frame (before the reference's 4x cross dilation)."""
    import numpy as np
    g = _gen(seed, f"video:{n}:{h}:{w}")
    yy = torch.linspace(0, 1, h).view(1, h, 1, 1)
    xx = torch.linspace(0, 1, w).view(1, 1, w, 1)
    tt = torch.arange(n, dtype=torch.float32).view(n, 1, 1, 1)
    ph = torch.rand((1, 1, 1, 3), generator=g) * 6.28
    base = 0.5 + 0.35 * torch.sin(6.28 * (2.0 * xx + 0.02 * tt) + ph) * torch.cos(6.28 * (1.5 * yy - 0.015 * tt))
    x = (base + 0.15 * (torch.rand((n, h, w, 3), generator=g) - 0.5)).clamp_(0, 1)
    frames = (x * 255).round().to(torch.uint8).numpy()
    masks = np.zeros((n, h, w), dtype=np.uint8)
    hh, ww = max(h // 3, 1), max(w // 4, 1)
    for i in range(n):
        y0 = int((h - hh) * (0.5 + 0.4 * math.sin(0.5 * i)))
        x0 = int((w - ww) * (i / max(n - 1, 1)))
        masks[i, y0:y0 + hh, x0:x0 + ww] = 1
    return frames, masks


def write_eval_dataset(root, videos, h=270, w=480, seed=0, dataset="davis"):
    """A synthetic dataset in the layout the reference's evaluate.py reads (core/dataset.py:82-135):
    ``<root>/<dataset>/test.json``, ``JPEGImages/<name>.zip`` of JPEG frames and ``test_masks/<name>/%05d.png``.
    ``videos`` is ``[(name, n_frames)]``.  Frames are smooth drifting colour waves at ``h`` x ``w`` (not 432x240, so
    the loader's resize matters); holes are a moving rectangle, and zip members are written out of order so the
    loader's sort matters.  Deterministic for a given seed, OpenCV and Pillow."""
    import json
    import os
    import zipfile
    import cv2
    import numpy as np
    base = os.path.join(root, dataset)
    os.makedirs(os.path.join(base, "JPEGImages"), exist_ok=True)
    yy = np.linspace(0, 1, h, dtype=np.float64)[:, None, None]
    xx = np.linspace(0, 1, w, dtype=np.float64)[None, :, None]
    for v, (name, n) in enumerate(videos):
        rng = np.random.default_rng([seed, v])
        ph = rng.uniform(0, 6.28, size=3)
        os.makedirs(os.path.join(base, "test_masks", name), exist_ok=True)
        with zipfile.ZipFile(os.path.join(base, "JPEGImages", f"{name}.zip"), "w") as z:
            for i in reversed(range(n)):
                img = 0.5 + 0.35 * np.sin(6.28 * (1.3 * xx + 0.7 * yy + 0.02 * i) + ph) * np.cos(6.28 * (0.9 * yy - 0.015 * i))
                ok, jpg = cv2.imencode(".jpg", cv2.cvtColor((img * 255).round().astype(np.uint8), cv2.COLOR_RGB2BGR))
                assert ok
                z.writestr(f"{i:05d}.jpg", jpg.tobytes())
        hh, ww = h // 6, w // 8
        for i in range(n):
            m = np.zeros((h, w), np.uint8)
            y0 = int((h - hh) * (0.5 + 0.4 * math.sin(0.5 * i + v)))
            x0 = int((w - ww) * (i / max(n - 1, 1)))
            m[y0:y0 + hh, x0:x0 + ww] = 255
            cv2.imwrite(os.path.join(base, "test_masks", name, f"{i:05d}.png"), m)
    with open(os.path.join(base, "test.json"), "w") as f:
        json.dump({name: n for name, n in videos}, f)
    return root
