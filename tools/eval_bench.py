"""Timing of the evaluation path on one GPU: ``metrics.psnr_ssim`` per frame, the fp64 numpy oracle on the host for
comparison, and ``evaluate.evaluate_video`` on a synthetic 60-frame 432x240 video with stress weights.

    python tools/eval_bench.py --out profiles/eval/eval_bench.json

(a) psnr_ssim: N = 1, 12, 60 frames of 432x240 (quarter-integer canvases, as evaluation produces), CUDA events
    around ``--iters`` calls after warm-up.  The calls rotate over enough input sets (> 256 MB in all) that the
    inputs are read from HBM, not from the 126 MB L2.  Bytes: H*W*3 * (1 + 4) per frame (uint8 original + fp32 canvas).
(b) oracle: ``oracle.restate_metrics.calc_psnr_and_ssim`` (scipy, fp64, one host thread per call) per frame.
(c) evaluate_video: total, ``VideoInpainter.composite`` and ``psnr_ssim`` times, CUDA events, after one warm-up
    video (which also captures the CUDA graphs).
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
H, W = 240, 432


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True)
    return dict(zip(q.split(","), [s.strip() for s in r.stdout.strip().split(",")])) if r.returncode == 0 else {}


def _inputs(n, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    a = torch.randint(0, 256, (n, H, W, 3), generator=g, device=dev, dtype=torch.uint8)
    d = torch.randint(-40, 41, (n, H, W, 3), generator=g, device=dev).float() / 4
    return a, (a.float() + d).clamp_(0, 255)


def bench_kernel(n, iters, dev):
    from e2fgvi_b200 import metrics
    per_set = n * H * W * 3 * 5
    sets = [_inputs(n, s, dev) for s in range(max(2, -(-256 * 2 ** 20 // per_set)))]
    for a, b in sets:
        metrics.psnr_ssim(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        a, b = sets[i % len(sets)]
        metrics.psnr_ssim(a, b)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    return dict(frames=n, input_sets=len(sets), input_bytes_total=per_set * len(sets), us_per_call=us,
                us_per_frame=us / n, bytes_per_frame=H * W * 3 * 5, achieved_GBps=per_set / us * 1e-3)


def bench_oracle(frames):
    from oracle import restate_metrics as RM
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    b = np.clip(a + rng.integers(-40, 41, a.shape) / 4, 0, 255).astype(np.float32)
    RM.calc_psnr_and_ssim(a, b)
    t = time.perf_counter()
    for _ in range(frames):
        RM.calc_psnr_and_ssim(a, b)
    return dict(frames=frames, ms_per_frame=(time.perf_counter() - t) * 1e3 / frames)


def bench_evaluate_video(n, reps, dev, model_name):
    import importlib
    from e2fgvi_b200 import evaluate as E
    from e2fgvi_b200 import metrics
    from e2fgvi_b200.synth import synth_state_dict, synth_video
    from e2fgvi_b200.video import VideoInpainter
    from oracle.restate_video import dilate_cross
    gen = importlib.import_module("e2fgvi_b200.model." + model_name).InpaintGenerator().eval()
    gen.load_state_dict(synth_state_dict(gen, "stress", 0), strict=True)
    gen.to(dev)
    vi = VideoInpainter(gen)
    frames, raw = synth_video(n, H, W, 3)
    frames = torch.from_numpy(frames).to(dev)
    masks = torch.from_numpy(np.stack([dilate_cross(m) for m in raw])).to(dev)
    E.evaluate_video(vi, frames, masks)                              # warm-up: graph capture, module load
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tot, comp_t, met_t = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        ev[0].record()
        comp = vi.composite(frames, masks)
        ev[1].record()
        p, s = metrics.psnr_ssim(frames, comp)
        ev[2].record()
        p.cpu(), s.cpu()
        torch.cuda.synchronize()
        tot.append((time.perf_counter() - t0) * 1e3)
        comp_t.append(ev[0].elapsed_time(ev[1]))
        met_t.append(ev[1].elapsed_time(ev[2]))
    total, composite, metric = float(np.median(tot)), float(np.median(comp_t)), float(np.median(met_t))
    return dict(model=model_name, weights="stress", frames=n, reps=reps, total_ms=total, composite_ms=composite,
                metric_ms=metric, metric_share=metric / total, ms_per_frame=total / n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--oracle_frames", type=int, default=10)
    ap.add_argument("--video_reps", type=int, default=5)
    ap.add_argument("--model", default="e2fgvi_hq")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench needs a GPU")
    from e2fgvi_b200 import build
    build.build()
    dev = torch.device("cuda:0")
    res = dict(gpu=gpu_info(), torch=torch.__version__, size=[H, W])
    res["psnr_ssim"] = [bench_kernel(n, args.iters, dev) for n in (1, 12, 60)]
    res["oracle_cpu"] = bench_oracle(args.oracle_frames)
    res["evaluate_video"] = bench_evaluate_video(60, args.video_reps, dev, args.model)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
