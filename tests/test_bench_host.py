"""CPU: host-side logic of bench.py (no GPU, no oracle run): the GPU arm and the reference arm of one workload must
print the SAME ``config`` object, input sets must exceed L2, every BASELINE config is a named workload."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_workload_table_covers_baseline_configs():
    import bench
    idx = sorted(v[6] for v in bench.WORKLOADS.values())
    assert idx == [1, 2, 3, 4]                      # configs[0] is the CPU reference arm itself
    for name, (_, H, W, T, l_t, B, _) in bench.WORKLOADS.items():
        assert H % 60 == 0 and W % 108 == 0 and 0 < l_t < T and B >= 1
        set_bytes = B * T * 3 * H * W * 4
        assert bench.n_input_sets(set_bytes) * set_bytes > bench.L2_BYTES, name
        cfg = bench.workload_config(name, B, 1)
        assert json.loads(json.dumps(cfg)) == cfg and "workload" in cfg and "model" not in cfg


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun only rank 0 runs the CPU arm; the others exit 0 without output or work."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_clock_sampler_keeps_only_samples_of_the_timed_region():
    """The nvidia-smi sampler starts before the warm-up (its attach must not land in the timed region) and filters its
    samples by their own timestamps; unknown timestamp formats and too-short regions fall back to all samples."""
    import datetime
    import time

    import bench

    def ts(t):
        return datetime.datetime.fromtimestamp(t).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]

    class FakeProc:
        def __init__(self, lines):
            self.lines = lines

        def terminate(self):
            pass

        def communicate(self, timeout=None):
            return "\n".join(self.lines), None

    now = time.time()
    idle = "Not Active, Not Active, Not Active, Not Active"
    capped = "Not Active, Not Active, Not Active, Active"
    s = bench.ClockSampler.__new__(bench.ClockSampler)
    s.p = FakeProc([f"{ts(now - 2.0)}, 1965, 1965, {idle}",          # warm-up sample: dropped
                    f"{ts(now - 0.3)}, 1650, 1965, {capped}", f"{ts(now - 0.1)}, 1640, 1965, {capped}"])
    s.t0 = now - 0.5
    got = s.stop()
    assert got == {"sm_mhz": 1645.0, "sm_max_mhz": 1965.0, "samples": 2, "reasons": ["sw_power_cap"]}
    s = bench.ClockSampler.__new__(bench.ClockSampler)
    s.p = FakeProc([f"{ts(now - 2.0)}, 1900, 1965, {idle}"])          # nothing inside the region: use what there is
    s.t0 = now - 0.01
    assert s.stop()["samples"] == 1
    s = bench.ClockSampler.__new__(bench.ClockSampler)
    s.p = FakeProc([f"Tue Sep 23 13:20:46 2026, 1700, 1965, {capped}"])   # unknown timestamp format: kept
    s.t0 = now - 0.5
    assert s.stop() == {"sm_mhz": 1700.0, "sm_max_mhz": 1965.0, "samples": 1, "reasons": ["sw_power_cap"]}


def test_dump_outputs_keep_small_arrays_and_sample_large_ones():
    """--dump-outputs: float32 arrays, small ones whole, a large one as the same seeded sample of distinct elements on
    every run, three sampled arrays within 64 MB."""
    import numpy as np
    import torch

    import bench
    assert 3 * bench.DUMP_SAMPLE * 4 <= 64 << 20
    pred = torch.arange(bench.DUMP_SAMPLE + 1000, dtype=torch.float32)     # value == flat index
    flows = (torch.ones(2, 3), torch.zeros(2, 3, dtype=torch.float64))
    a, b = bench.output_arrays(pred, flows), bench.output_arrays(pred, flows)
    assert sorted(a) == ["flows_backward", "flows_forward", "pred_sample"]
    assert all(v.dtype == np.float32 for v in a.values()) and a["flows_forward"].shape == (2, 3)
    s = a["pred_sample"]
    assert s.shape == (bench.DUMP_SAMPLE,) and np.array_equal(s, b["pred_sample"]) and np.all(np.diff(s) > 0)
