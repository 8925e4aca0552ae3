#!/usr/bin/env python
"""bench.py — frames/sec of InpaintGenerator.forward on synthetic 432x240 5+3 clips (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--clips-per-gpu B] [--workload W]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (N > 1, one rank per GPU, NCCL)

Headline: a step = one forward over B clips per GPU (default 8 = BASELINE configs[3]'s per-GPU share: 64 clips over
8 GPUs) followed, for N > 1, by the single all-gather output stitch (asynchronous, overlapped with the next step's
forward).  The same JSON line also carries, as first-class fields, the other BASELINE configs measured in the same
process: ``workloads.b1`` (configs[1]: ONE 432x240 5+3 clip per call, eager and CUDA-graph), ``workloads.hq720``
(configs[2]) and ``workloads.hq1080`` (configs[4], one clip per GPU).  Prints ONE JSON line on rank 0.
"""
import argparse
import importlib
import datetime
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: the benchmark writes nothing into it

import torch  # noqa: E402

# BASELINE.json configs.  name -> (model module, H, W (mirror-padded to multiples of 60 / 108 like test.py:156-165),
# T, l_t, clips per GPU per step, BASELINE config index)
WORKLOADS = {
    "base": ("model.e2fgvi", 240, 432, 8, 5, 8, 3),          # configs[3] per-GPU share (64 clips over 8 GPUs)
    "b1": ("model.e2fgvi", 240, 432, 8, 5, 1, 1),            # configs[1]: one clip per call
    "hq720": ("model.e2fgvi_hq", 720, 1296, 8, 5, 1, 2),     # configs[2]: 720x1280, 5+3
    "hq1080": ("model.e2fgvi_hq", 1080, 1944, 16, 10, 1, 4),  # configs[4]: 1080x1920, 10+6, one clip per GPU
}
L2_BYTES = 126e6


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def host_cores():
    """CPU threads this process may really use: min(affinity mask, cgroup cpu quota) — os.cpu_count() alone
    reports the host's cores inside a quota-limited container and oversubscribes the oracle by 10-100x."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md).

    The process is started BEFORE the warm-up steps: nvidia-smi needs 0.1-0.5 s to attach to the driver and, while it
    does, kernel launches of this process stall behind it — started right in front of the timed region (as this file
    did until run 27 of round 2) that cost landed inside the measurement: 36.6-38.0 ms per step in the device-resident
    loop against 34.2-34.9 ms in the end-to-end loop two seconds later, with only 1-3 samples returned.  Every line
    carries nvidia-smi's own timestamp; only the samples between ``mark_start()`` and ``stop()`` are used."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        self.t0 = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def mark_start(self):
        self.t0 = time.time()

    def stop(self):
        t1 = time.time()
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
            out, _ = self.p.communicate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []                                           # (inside the timed region?, sm, max sm, active reasons)
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm_v, mx_v = float(f[1]), float(f[2])
            except ValueError:
                continue
            inside = True
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                inside = self.t0 is None or (self.t0 - 0.05 <= ts <= t1 + 0.05)
            except ValueError:
                pass                                        # unknown timestamp format: keep the sample
            rows.append((inside, sm_v, mx_v, [n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")]))
        used = [r for r in rows if r[0]] or rows            # a timed region shorter than one sampling period: use all
        sm, mx = [r[1] for r in used], [r[2] for r in used]
        reasons = {n for r in used for n in r[3]}
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_model(device, module="model.e2fgvi"):
    net = importlib.import_module(module)
    from e2fgvi_b200.synth import synth_state_dict
    model = net.InpaintGenerator().eval()
    sd = synth_state_dict(model, "default", 0)          # the reference's own init family (BASELINE config)
    model.load_state_dict(sd, strict=True)
    return (model.to(device) if device is not None else model), sd


DUMP_SAMPLE = 1 << 22     # elements kept of a larger output array: three arrays stay under 64 MB of float32


def output_arrays(pred, flows):
    """What ``model(x, l_t)`` returned, as float32 host arrays for ``--dump-outputs``.  An array of more than
    ``DUMP_SAMPLE`` elements is replaced by ``<name>_sample``: the elements at ``DUMP_SAMPLE`` distinct flat indices
    drawn by ``torch.randperm`` from a CPU generator seeded with 0, in increasing index order."""
    out = {}
    for name, t in (("pred", pred), ("flows_forward", flows[0]), ("flows_backward", flows[1])):
        t = t.detach().float()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        out[name] = t.cpu().numpy()
    return out


def workload_config(name, B, world, precision="strict"):
    """The ``config`` object of the JSON line — IDENTICAL for the GPU arm and the reference arm of one workload."""
    module, H, W, T, l_t, _, idx = WORKLOADS[name]
    set_mb = B * T * 3 * H * W * 4 / 1e6
    return {"workload": f"{module.split('.')[-1]} {W}x{H}" + (" (mirror-padded)" if name.startswith("hq") else "")
                        + f", {l_t} local + {T - l_t} ref frames, {B} clip(s) per GPU per step (BASELINE configs[{idx}]"
                        + (" per-GPU share)" if name == "base" else ")"),
            "global_batch_clips": B * world, "frames_per_clip": T, "parallelism": f"clip-dp{world}",
            "l2": f"inputs rotate over {n_input_sets(set_mb * 1e6)} sets x {set_mb:.0f} MB (> 126 MB L2)",
            "precision": precision,
            "weights": "random-init, reference default family (e2fgvi_b200.synth 'default', seed 0)"}


def n_input_sets(set_bytes):
    return max(2, min(32, math.ceil(1.3 * L2_BYTES / set_bytes)))


def metric_name(name):
    _, H, W, T, l_t, _, _ = WORKLOADS[name]
    base = f"frames/sec InpaintGenerator.forward {W}x{H}x({l_t}+{T - l_t})"
    return base if name == "base" else base + f" [{name}]"


def cpu_oracle_fps(sd, name="base", steps=1, warmup=0):
    """The reference's CPU implementation of the path: the oracle port (oracle/restate.py) on all host threads,
    ONE clip of the workload's shape per step (the reference itself is single-process, b=1: test.py:108,152-166;
    clips are independent, so its frames/s does not depend on how many clips a step holds)."""
    from e2fgvi_b200.synth import synth_frames
    from oracle import restate
    _, H, W, T, l_t, _, _ = WORKLOADS[name]
    torch.set_num_threads(host_cores())
    x = synth_frames(1, T, H, W, seed=3)
    with torch.no_grad():
        for _ in range(warmup):
            restate.inpaint_generator_forward(sd, x, l_t)
        t0 = time.perf_counter()
        for _ in range(steps):
            restate.inpaint_generator_forward(sd, x, l_t)
        dt = time.perf_counter() - t0
    return steps * T / dt, dt / steps, torch.get_num_threads()


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port; /root/reference does not exist on the GPU box), on
    the SAME config object as the GPU arm.  Each step is a bounded sample of the workload: one of its clips."""
    if rank != 0:
        return
    name = args.workload
    module, H, W, T, l_t, default_b, _ = WORKLOADS[name]
    B = args.clips_per_gpu or default_b
    _, sd = make_model(None, module)
    steps, warmup = args.steps, args.warmup
    if name.startswith("hq"):               # 65 s (720p) .. minutes (1080p) per clip on a CPU: one clip, no warm-up
        steps, warmup = 1, 0
    fps, s_per_step, cores = cpu_oracle_fps(sd, name, steps=steps, warmup=warmup)
    line = {
        "impl": "reference", "metric": metric_name(name), "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, B, world, args.precision),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} step(s), each ONE clip of the workload's {B} per GPU ({T} frames {W}x{H}; "
                                   "clips are independent, so CPU frames/s does not depend on the clips per step): "
                                   "oracle/restate.py, torch CPU fp32 on all host threads; DCN = explicit "
                                   "restatement (mmcv is not installable offline)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ops._timed name -> (kernel name, roofline that bounds it, tensor-work multiplier)
KINDS = {"focal_window_attention": ("focal_attn_kernel", "tensor", 1.0),
         "deform_align_fused": ("dcn_kernel", "tensor", 1.0),
         # bf16x3 kernels: algorithmic fp32 FLOPs; each costs 3 bf16 MMAs, so <= 1/3 of the bf16 peak
         "conv3x3_bf16x3": ("conv3x3_kernel", "tensor", 3.0),
         "linear_bf16x3": ("linear_kernel", "tensor", 3.0),
         "t2t_fold_unfold": ("t2t_fold733_kernel", "hbm", 1.0),
         "t2t_fold": ("t2t_fold_kernel", "hbm", 1.0), "t2t_unfold": ("t2t_unfold733_kernel", "hbm", 1.0),
         "layernorm_split": ("layernorm_split_kernel", "hbm", 1.0),
         "upsample2x_split": ("upsample2x_split_kernel", "hbm", 1.0),
         "window_pool": ("window_pool_kernel", "hbm", 1.0), "pack_rows": ("pack_rows_kernel", "hbm", 1.0)}


def kernel_rooflines(prof, total_ms, traffic):
    """Per-kernel live timing (CUDA events around each launch inside the timed region) -> roofline entries."""
    hbm, _, tf_sust, _ = peaks()
    kernels = {}
    for key, (kname, bound, mult) in KINDS.items():
        ev = prof.get(key, [])
        if not ev:
            continue
        durs = [a.elapsed_time(b) for a, b, _ in ev]
        work = sum(w for _, _, w in ev)
        tot_ms = sum(durs)
        if bound == "tensor":
            ach, peak, unit = work / (tot_ms * 1e-3) / 1e12, tf_sust, "TFLOP/s"
        else:
            ach, peak, unit = work / (tot_ms * 1e-3) / 1e9, hbm, "GB/s"
        kernels[kname] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                          "launches_timed": len(durs), "avg_launch_ms": tot_ms / len(durs),
                          "share_of_step": tot_ms / total_ms, "traffic": (traffic or {}).get(kname)}
        if mult != 1.0:
            kernels[kname]["tensor_work_multiplier"] = mult
            kernels[kname]["tensor_pipe_frac"] = mult * ach / peak
    return kernels


def dominant(kernels):
    if not kernels:
        return None
    _, _, _, src = peaks()
    dom = max(kernels, key=lambda k: kernels[k]["share_of_step"])
    return dict(kernels[dom], kernel=dom,
                peak_source=f"{src} " + ("bf16_tflops_sustained" if kernels[dom]["bound"] == "tensor" else "hbm_gbs"),
                note="achieved = algorithmic work (SURVEY 8d) / live CUDA-event launch time inside the timed region")


class Measurement:
    """One workload on this rank's GPU: device-resident timing (value), per-kernel live timing, end-to-end timing
    through the public API with pinned HOST buffers (H2D of the inputs and D2H of the result inside the timed region)."""

    def __init__(self, name, model, dev, rank, world, B, steps, warmup):
        from e2fgvi_b200 import clips as C
        from e2fgvi_b200.synth import synth_frames
        self.C = C
        self.name, self.model, self.dev, self.rank, self.world = name, model, dev, rank, world
        _, self.H, self.W, self.T, self.l_t, _, _ = WORKLOADS[name]
        self.B, self.steps, self.warmup = B, steps, max(warmup, 3)
        set_bytes = B * self.T * 3 * self.H * self.W * 4
        self.n_sets = n_input_sets(set_bytes)
        self.host_sets = [synth_frames(B, self.T, self.H, self.W, seed=100 + rank * 32 + i).pin_memory()
                          for i in range(self.n_sets)]
        self.dev_sets = [h.to(dev) for h in self.host_sets]
        self.out_host = torch.empty((B * self.T, 3, self.H, self.W), dtype=torch.float32).pin_memory()
        self.num_clips = B * world
        self.stitch = C.make_stitcher(self.num_clips, self.T, rank, world, device=self.dev)   # peer-memory pushes on one NVLink box
        self._copy_streams = None
        self._dev_in = None

    def sync(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def _loop(self, n, inputs, to_host=False, stitch=True):
        """n steps; the stitch of step i overlaps the forward of step i+1 (double-buffered landing zone).

        ``to_host``: the end-to-end pipeline a caller of the public API runs — every step's inputs come from PINNED HOST
        memory and its result goes back to pinned host memory, inside the timed region.  The copies ride their own
        streams: the H2D of step i+1 is issued while step i computes (double-buffered device input), the D2H of step i
        runs while step i+1 computes; the forward itself is the unchanged ``model(x, l_t)`` call on the current stream."""
        pending = None
        B, T = self.B, self.T
        main = torch.cuda.current_stream()
        if to_host and self._copy_streams is None:
            self._copy_streams = (torch.cuda.Stream(device=self.dev), torch.cuda.Stream(device=self.dev))
        h2d, d2h = self._copy_streams if to_host else (None, None)

        if to_host and self._dev_in is None:                # two device input buffers, refilled in place (no allocation
            self._dev_in = [torch.empty_like(inputs[0], device=self.dev) for _ in range(2)]   # inside the timed loop)
        consumed = [None, None]                             # event: the forward that read buffer j has been enqueued on `main`
        landed = []                                         # events: result of step i is on the host

        def upload(i):
            j = i % 2
            with torch.cuda.stream(h2d):
                if consumed[j] is not None:
                    h2d.wait_event(consumed[j])             # step i-2 has read this buffer
                self._dev_in[j].copy_(inputs[i % self.n_sets], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(h2d)
            return self._dev_in[j], ev

        def download(t):
            """device tensor produced on `main` -> pinned host, on the D2H stream"""
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(d2h):
                d2h.wait_event(ev)
                self.out_host.copy_(t, non_blocking=True)
                done = torch.cuda.Event()
                done.record(d2h)
            t.record_stream(d2h)
            landed.append(done)

        nxt_in = upload(0) if to_host and n > 0 else None
        for i in range(n):
            if to_host:
                x, ev = nxt_in
                main.wait_event(ev)
                if len(landed) > 2:
                    # bounded queue depth, as a real caller would run it: the host never runs more than three results ahead
                    # (the device still has two steps queued, so this wait costs no device time; without it the caching
                    # allocator keeps growing the pool of in-flight 80 MB results and cudaMalloc synchronises the device)
                    landed[len(landed) - 3].synchronize()
            else:
                x = inputs[i % self.n_sets]
            pred, flows = self.model(x, self.l_t)
            if to_host:
                consumed[i % 2] = torch.cuda.Event()
                consumed[i % 2].record(main)
            if to_host and i + 1 < n:
                nxt_in = upload(i + 1)                    # overlaps this step's forward
            if to_host and self.world > 1:
                main.wait_stream(d2h)                     # the landing buffer about to be reused has been read out
            nxt = self.stitch.start(pred) if (self.world > 1 and stitch) else None
            if pending is not None:
                got = pending.wait()
                if to_host:
                    download(got[self.rank * B * T:(self.rank + 1) * B * T])
            if self.world == 1 and to_host:
                download(pred)
            pending = nxt
        if pending is not None:
            got = pending.wait()
            if to_host:
                download(got[self.rank * B * T:(self.rank + 1) * B * T])
        if to_host:
            main.wait_stream(d2h)                          # the timed region ends when the last result is on the host
        return (pred, flows) if n > 0 else None

    def run(self, sample_clocks=False, profile=True, keep_outputs=False):
        from e2fgvi_b200 import ops
        res = {}
        with torch.no_grad():
            sampler = ClockSampler(self.dev.index) if (sample_clocks and self.rank == 0) else None
            self._loop(self.warmup, self.dev_sets)
            self.sync()
            n0 = ops.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.sync()
            if sampler:
                sampler.mark_start()
            e0.record()
            last = self._loop(self.steps, self.dev_sets)
            e1.record()
            self.sync()
            res["launches"] = ops.launch_count() - n0
            res["outputs"] = output_arrays(*last) if keep_outputs and last else None
            del last
            res["clocks"] = sampler.stop() if sampler else None
            ms = e0.elapsed_time(e1)
            ms_free = ms
            if self.world > 1:
                # diagnosis of the scaling loss: the same steps WITHOUT the stitch — every rank runs free, so the max over
                # ranks is the slowest GPU's own time (boards differ by a few % under the power cap) and the difference to
                # the stitched loop is what the exchange itself costs
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                self._loop(self.steps, self.dev_sets, stitch=False)
                g1.record()
                self.sync()
                ms_free = g0.elapsed_time(g1)
            # ---- per-kernel live timing in a SEPARATE pass over the same steps: two CUDA events per launch cost host time
            #      that would distort a launch-bound workload (one clip per call) if it ran inside the region above
            prof, ms_prof = None, None
            if profile:
                saved_graphs = getattr(self.model, "_graphs", None)
                saved_overlap = getattr(self.model, "overlap_flow", False)
                self.model.overlap_flow = False         # concurrent streams would inflate each other's event-timed launches
                if saved_graphs is not None:
                    self.model._graphs = None           # kernels inside a replayed graph cannot be timed one by one
                    self._loop(2, self.dev_sets)
                    self.sync()
                prof = ops.profile_kernels(True)
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                self._loop(self.steps, self.dev_sets)
                p1.record()
                self.sync()
                ops.profile_kernels(False)
                ms_prof = p0.elapsed_time(p1)
                if saved_graphs is not None:
                    self.model._graphs = saved_graphs
                self.model.overlap_flow = saved_overlap
            # ---- end to end through the public API with HOST buffers
            self._loop(2, self.host_sets, to_host=True)
            self.sync()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            self._loop(self.steps, self.host_sets, to_host=True)
            f1.record()
            self.sync()
            ms_e2e = f0.elapsed_time(f1)
        t = torch.tensor([ms, ms_e2e, ms_free], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            per_rank = [torch.zeros_like(t) for _ in range(self.world)]
            torch.distributed.all_gather(per_rank, t)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            res["ranks"] = {"ms_per_step": [float(x[0]) / self.steps for x in per_rank],
                            "ms_per_step_without_stitch": [float(x[2]) / self.steps for x in per_rank],
                            "stitch_cost_ms_per_step": (float(t[0]) - float(t[2])) / self.steps,
                            "note": "value uses the max over ranks of the stitched loop; without the stitch every rank runs "
                                    "free, so its max is the slowest board's own time"}
        ms, ms_e2e = float(t[0]), float(t[1])
        frames = self.num_clips * self.T * self.steps
        nbytes = self.B * self.T * 3 * self.H * self.W * 4 * self.world
        res.update(ms=ms, ms_per_step=ms / self.steps, value=frames / (ms * 1e-3), prof=prof, ms_prof=ms_prof,
                   e2e={"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": nbytes,
                        "d2h_bytes_per_step": nbytes, "ms_per_step": ms_e2e / self.steps})
        log(f"{self.name}: {res['ms_per_step']:.2f} ms/step device, {ms_e2e / self.steps:.2f} ms/step e2e")
        return res

    def free(self):
        self.host_sets = self.dev_sets = self.out_host = self._dev_in = None
        if hasattr(self.stitch, "close"):
            self.stitch.close()                  # peer-memory landing buffers are cudaMalloc'd outside torch's allocator
        torch.cuda.empty_cache()


def traffic_for(name):
    """DRAM bytes per launch from the committed `ncu` step capture of THIS workload (profiles/ncu_traffic.json,
    keyed by workload); None for workloads without a capture (never the bytes of another shape)."""
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(tpath):
        return None
    d = json.load(open(tpath))
    return d.get(name) if isinstance(d.get(name), dict) else None


def graph_latency(model, one, l_t, reps=10):
    from e2fgvi_b200.graph import GraphedGenerator
    graphed = GraphedGenerator(model, one, l_t)
    for _ in range(3):
        graphed(one)
    torch.cuda.synchronize()
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record()
    for _ in range(reps):
        graphed(one)
    h1.record()
    torch.cuda.synchronize()
    return h0.elapsed_time(h1) / reps


def video_driver_run(model, H, W):
    """test.py's sliding-window loop (SURVEY 8(f) rank 4) on a synthetic 60-frame video, pinned uint8 host -> host."""
    import numpy as np
    from e2fgvi_b200.synth import synth_video
    from e2fgvi_b200.video import VideoInpainter
    vf, vm = synth_video(60, H, W, 21)
    vf_t, vm_t = torch.from_numpy(vf).pin_memory(), torch.from_numpy(vm).pin_memory()
    drv = VideoInpainter(model, clips_per_call=4)
    drv(vf_t, vm_t)
    torch.cuda.synchronize()          # rank-0-only section: no collective
    v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    v0.record()
    comp = drv(vf_t, vm_t).cpu()
    v1.record()
    torch.cuda.synchronize()
    ms_v = v0.elapsed_time(v1)
    sched = drv.schedule(60)
    net_frames = sum(len(nb) + len(rf) for _, nb, rf in sched)
    return {"video_frames": 60, "windows": len(sched), "network_frames": net_frames, "ms": ms_v,
            "video_frames_per_s": 60 / (ms_v * 1e-3), "network_frames_per_s": net_frames / (ms_v * 1e-3),
            "untouched_pixels_exact": bool(np.array_equal(comp.numpy()[vm == 0], vf[vm == 0]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips-per-gpu", type=int, default=None)
    ap.add_argument("--workload", default="base", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-workloads", action="store_true",
                    help="skip the b1 / hq720 / hq1080 / video-driver sections of the default run")
    ap.add_argument("--precision", default="strict", choices=["strict", "tf32"],
                    help="library op precision (only matters for the few remaining torch glue ops)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload returned (rank 0) as DIR/<name>.npy, "
                         "float32; inputs and weights are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)

    from e2fgvi_b200 import clips as C
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return
    rank, world, local_rank = C.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    from e2fgvi_b200 import build as _build
    _build.build()
    name = args.workload
    module, H, W, T, l_t, default_b, _ = WORKLOADS[name]
    B = args.clips_per_gpu or default_b
    models = {}

    def get_model(mod):
        if mod not in models:
            models[mod] = make_model(dev, mod)
            models[mod][0].precision = args.precision
        return models[mod]

    model, sd = get_model(module)
    log(f"rank {rank}/{world}: model ready, workload={name}, host cores={host_cores()}")
    head = Measurement(name, model, dev, rank, world, B, args.steps, args.warmup)
    stitch_kind = ("none (one GPU)" if world == 1 else
                   "peer-memory DMA pushes + stream-memop flags (clips.PeerStitcher)" if type(head.stitch).__name__ == "PeerStitcher"
                   else "all_gather_into_tensor (clips.ClipStitcher)")
    main_res = head.run(sample_clocks=True, keep_outputs=args.dump_outputs is not None and rank == 0)
    if main_res["outputs"] is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for oname, arr in main_res.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, oname + ".npy"), arr)
        log(f"outputs of the last timed step written to {args.dump_outputs}")
    kernels = kernel_rooflines(main_res["prof"], main_res["ms_prof"], traffic_for(name)) if rank == 0 else {}
    one_clip = head.dev_sets[0][:1].clone()
    head.free()

    extra, b1 = {}, None
    video = None
    if not args.no_extra_workloads and name == "base":
        # ---- BASELINE configs[1] / [2] / [4] in the same process (every rank runs them; whole-job aggregate)
        for wname in ("b1", "hq720", "hq1080"):
            wmod, wH, wW, wT, wl_t, wB, _ = WORKLOADS[wname]
            try:
                wm, _ = get_model(wmod)
                steps = {"b1": 20, "hq720": 5, "hq1080": 3}[wname]
                m = Measurement(wname, wm, dev, rank, world, wB, steps, 3)
                eager = None
                if wname == "b1":
                    # one clip per call is launch-bound from Python (~200 launches for ~6 ms of GPU work): measured
                    # eagerly first, then — the number reported as `value` — with model.enable_cuda_graphs(), i.e. the
                    # same public call model(x, l_t) replaying a per-shape captured CUDA graph
                    r0 = m.run(profile=False)
                    eager = {"value": r0["value"], "ms_per_step": r0["ms_per_step"], "e2e": r0["e2e"]}
                    wm.enable_cuda_graphs(True)
                r = m.run()
                if wname == "b1":
                    wm.enable_cuda_graphs(False)
                entry = {"metric": metric_name(wname), "value": r["value"], "unit": "frames/s", "steps": steps, "warmup": 3,
                         "ms_per_step": r["ms_per_step"], "e2e": r["e2e"], "gpu_launches": r["launches"],
                         "config": workload_config(wname, wB, world, args.precision)}
                if eager is not None:
                    entry["config"]["cuda_graphs"] = "model.enable_cuda_graphs(): the public call replays a captured graph"
                    entry["eager"] = eager
                if rank == 0:
                    wk = kernel_rooflines(r["prof"], r["ms_prof"], traffic_for(wname))
                    entry["roofline"] = dominant(wk)
                    entry["roofline_kernels"] = wk
                if wname == "b1" and world == 1:
                    try:                              # bare replay of one captured graph on a device-resident input
                        entry["cuda_graph_ms_per_step"] = graph_latency(wm, one_clip, wl_t)
                        entry["cuda_graph_value"] = wT / (entry["cuda_graph_ms_per_step"] * 1e-3)
                    except Exception as exc:      # reported, never fatal for the headline numbers
                        log(f"CUDA-graph latency run failed: {exc!r}")
                m.free()
                extra[wname] = entry
            except Exception as exc:
                log(f"workload {wname} failed: {exc!r}")
                extra[wname] = {"error": repr(exc)}
        b1 = extra.get("b1")
        if rank == 0:
            try:
                video = video_driver_run(model, H, W)
            except Exception as exc:
                log(f"video driver run failed: {exc!r}")

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and name in ("base", "b1"):
            log("timing the CPU oracle (1 warm-up + 2 clips) ...")
            fps, s_per, cores = cpu_oracle_fps(sd, name, steps=2, warmup=1)
            log(f"CPU oracle: {s_per:.2f} s/clip on {cores} threads")
            cpu = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                   "sample": "2 x one 5+3 clip forward after 1 warm-up (oracle/restate.py, torch CPU fp32; clips are "
                             "independent, so CPU frames/s does not depend on the clips per step)"}
        line = {
            "metric": metric_name(name), "value": main_res["value"], "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": head.warmup, "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate (DCN, attention kernels); bf16 3-term split operands / f32 "
                     "accumulate = fp32-level accuracy (conv, linear kernels)",
            "data": "synthetic", "config": workload_config(name, B, world, args.precision),
            "e2e": main_res["e2e"], "gpu_launches": main_res["launches"], "clocks": main_res["clocks"],
            "roofline": dominant(kernels), "roofline_kernels": kernels, "cpu_baseline": cpu,
            # BASELINE configs[1] (one clip per call) as first-class numbers next to the batched headline
            "fps_b1": None if not b1 or "value" not in b1 else b1["value"],
            "latency_b1_ms": None if not b1 or "ms_per_step" not in b1 else b1["ms_per_step"],
            "fps_b1_e2e": None if not b1 or "e2e" not in b1 else b1["e2e"]["value"],
            "fps_b1_eager": None if not b1 or "eager" not in b1 else b1["eager"]["value"],
            "fps_b1_cuda_graph": None if not b1 else b1.get("cuda_graph_value"),
            "latency_b1_cuda_graph_ms": None if not b1 else b1.get("cuda_graph_ms_per_step"),
            "speedup_vs_cpu_b1": None if not (b1 and cpu and "value" in b1) else b1["value"] / cpu["value"],
            "workloads": extra, "video_driver": video, "stitch": stitch_kind, "ranks": main_res.get("ranks"),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
