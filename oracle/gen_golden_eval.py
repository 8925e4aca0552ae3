"""TEST INFRASTRUCTURE — runs the UNMODIFIED ``/root/reference/evaluate.py`` (its ``main_worker``) on a synthetic
DAVIS-layout dataset in the build container and stores what it computed, as the golden for
``e2fgvi_b200.evaluate`` and ``e2f_psnr_ssim``.

    python -m oracle.gen_golden_eval        # only where /root/reference exists

How the script is made to run offline without touching it: ``matplotlib`` (imported by core/utils.py, unused here)
is replaced by ``unittest.mock`` modules, ``mmcv`` comes from ``oracle/mmcv_shim`` and ``skimage.measure.compare_ssim``
from ``oracle/skimage_shim`` (backed by ``oracle/restate_metrics.py``; scikit-image cannot be installed offline).
``init_i3d_model`` / ``calculate_i3d_activations`` / ``calculate_vfid`` are stubbed in ``core.metrics`` before the
script runs (the I3D weights are not shipped), ``calc_psnr_and_ssim`` and ``TestDataset.load_item`` are wrapped to
record what they saw, and ``InpaintGenerator.forward`` to record each window's clip and output.

Stored per case in ``tests/golden/<case>.npz`` (inputs are regenerated from seeds by
``e2fgvi_b200.synth.write_eval_dataset`` / ``synth_state_dict``):

* ``frames_sha256`` of the frames TestDataset loaded per video, and the dilated masks it loaded (bit-packed);
* ``canvas4_delta`` = 4 * canvas - 4 * frame as int16: the fp32 canvas calc_psnr_and_ssim scored (exact: every canvas
  value is a multiple of 1/4 at neighbor_stride 5), stored as a difference from the frame so it compresses;
* ``psnr`` / ``ssim`` per frame (fp64) and the metrics file text;
* evaluate.py's window schedule (``get_ref_index`` in its window loop) for video lengths 1..60;
* the network replay: SHA-256 of every window's clip, its local frame count, and the uint8 value of every hole pixel
  of its local frames, the only part of the network output the composite reads (evaluate.py:101-111).

The loaded frames themselves (about 2 MB per 10 frames compressed) are not stored: their hashes pin the regenerated
dataset.
"""
import os
import pickle
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")

# name -> (model, weight family, weight seed, dataset seed, [(video, frames)])
CASES = {
    "eval_e2fgvi": ("e2fgvi", "stress", 3, 21, [("bear", 11), ("car-turn", 7)]),
    "eval_hq": ("e2fgvi_hq", "stress", 4, 22, [("swan", 16)]),
}

CHILD = r'''
import sys, os, runpy, hashlib, pickle, importlib
from unittest import mock
import numpy as np
mmcv_shim, sk_shim, ref, tmp, out, model_name = sys.argv[1:7]
argv = sys.argv[7:]
sys.path[:] = [mmcv_shim, sk_shim, ref] + [p for p in sys.path if p not in ("", os.getcwd())]
for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation", "matplotlib.patches", "matplotlib.path"):
    sys.modules[name] = mock.MagicMock(name=name)
import core.metrics as M
import core.dataset as D
net = importlib.import_module("model." + model_name)
assert os.path.abspath(net.__file__).startswith(os.path.abspath(ref))
M.init_i3d_model = lambda: None
M.calculate_i3d_activations = lambda v1, v2, model, device=None: (np.zeros(1), np.zeros(1))
M.calculate_vfid = lambda real, fake: 0.0
rec = dict(loaded=[], scored=[], forward=[])
_calc = M.calc_psnr_and_ssim
def calc(img1, img2):
    p, s = _calc(img1, img2)
    rec["scored"].append((np.array(img1), np.array(img2), float(p), float(s)))
    return p, s
M.calc_psnr_and_ssim = calc
_load = D.TestDataset.load_item
def load_item(self, index):
    item = _load(self, index)
    rec["loaded"].append((item[2], np.stack(item[3]), item[1][:, 0].numpy().astype(np.uint8)))
    return item
D.TestDataset.load_item = load_item
_forward = net.InpaintGenerator.forward
def forward(self, masked_frames, num_local_frames):
    pred, flows = _forward(self, masked_frames, num_local_frames)
    u8 = (((pred + 1) / 2).cpu().permute(0, 2, 3, 1).numpy() * 255).astype(np.uint8)[:num_local_frames]
    rec["forward"].append((hashlib.sha256(masked_frames.cpu().numpy().tobytes()).hexdigest(), num_local_frames, u8))
    return pred, flows
net.InpaintGenerator.forward = forward
os.chdir(tmp)                       # the script writes ./results/
sys.argv = [os.path.join(ref, "evaluate.py")] + argv
glb = runpy.run_path(os.path.join(ref, "evaluate.py"), run_name="__main__")
# the script's reference-frame schedule (evaluate.py:22-28 with the loop of :86-91) for lengths 1..60
rec["schedule"] = {n: [(f, nb, glb["get_ref_index"](nb, n)) for f in range(0, n, glb["neighbor_stride"])
                       for nb in [list(range(max(0, f - glb["neighbor_stride"]),
                                             min(n, f + glb["neighbor_stride"] + 1)))]] for n in range(1, 61)}
with open(os.path.join(tmp, "results", f"{model_name}_davis", f"{model_name}_davis_metrics.txt")) as f:
    rec["metrics_txt"] = f.read()
with open(out, "wb") as f:
    pickle.dump(rec, f)
print("recorded", len(rec["scored"]), "frames,", len(rec["forward"]), "windows")
'''


def main(names=None):
    import hashlib
    import importlib
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    from e2fgvi_b200.evaluate import load_test_video
    from e2fgvi_b200.synth import synth_state_dict, write_eval_dataset
    from oracle import restate_metrics as RM
    from oracle import restate_video as RV
    from oracle.reference_loader import REFERENCE_ROOT, SHIM
    sk_shim = os.path.join(ROOT, "oracle", "skimage_shim")
    os.makedirs(OUT, exist_ok=True)
    for name, (model, family, wseed, dseed, videos) in CASES.items():
        if names and name not in names:
            continue
        with tempfile.TemporaryDirectory() as tmp:
            data = write_eval_dataset(os.path.join(tmp, "data"), videos, seed=dseed)
            mine = importlib.import_module("e2fgvi_b200.model." + model).InpaintGenerator()
            torch.save(synth_state_dict(mine, family, wseed), os.path.join(tmp, "ckpt.pth"))
            child = os.path.join(tmp, "child.py")
            with open(child, "w") as f:
                f.write(CHILD)
            rec_path = os.path.join(tmp, "rec.pkl")
            argv = ["--dataset", "davis", "--data_root", data, "--model", model, "--ckpt",
                    os.path.join(tmp, "ckpt.pth"), "--num_workers", "0"]
            subprocess.check_call([sys.executable, child, SHIM, sk_shim, REFERENCE_ROOT, tmp, rec_path, model] + argv,
                                  cwd=tmp)
            with open(rec_path, "rb") as f:
                rec = pickle.load(f)
            # our loader against the reference TestDataset, and our oracle driver + metrics against the script
            frames_all, masks_all, hashes = [], [], []
            for (vname, n), (lname, frames, masks) in zip(videos, rec["loaded"]):
                assert lname == vname and len(frames) == n
                f2, m2 = load_test_video(data, "davis", vname)
                assert np.array_equal(f2, frames) and np.array_equal(m2, masks), "load_test_video != TestDataset"
                frames_all.append(frames)
                masks_all.append(masks)
                hashes.append(hashlib.sha256(frames.tobytes()).hexdigest())
        frames = np.concatenate(frames_all)
        masks = np.concatenate(masks_all)
        comp = np.stack([s[1].astype(np.float32) for s in rec["scored"]])
        assert np.array_equal(np.stack([s[0] for s in rec["scored"]]), frames)
        assert np.array_equal(comp * 4, np.round(comp * 4)) and comp.min() >= 0 and comp.max() <= 255
        psnr = np.array([s[2] for s in rec["scored"]])
        ssim = np.array([s[3] for s in rec["scored"]])
        clips, l_ts, holes = [], [], []
        k, start = 0, 0
        for (vname, n), fr, ms in zip(videos, frames_all, masks_all):
            sched = RV.window_schedule(n)
            replay = rec["forward"][k:k + len(sched)]
            for (sha, l_t, u8), (_, nb, _) in zip(replay, sched):
                clips.append(sha)
                l_ts.append(l_t)
                holes.append(u8[ms[nb].astype(bool)])
            k += len(sched)
            mine_canvas = np.stack([c.astype(np.float32) for c in RV.inpaint_video(
                _replay_net(replay, ms), fr, ms)])
            assert np.array_equal(mine_canvas, comp[start:start + n]), "oracle driver != evaluate.py canvas"
            start += n
        assert k == len(rec["forward"])
        for i in range(len(comp)):
            p, s = RM.calc_psnr_and_ssim(frames[i], comp[i])
            assert p == psnr[i] and s == ssim[i]
        delta = (comp * 4).astype(np.int32) - frames.astype(np.int32) * 4
        np.savez_compressed(os.path.join(OUT, name + ".npz"), names=np.array([v for v, _ in videos]),
                            lengths=np.array([n for _, n in videos]), frames_sha256=np.array(hashes),
                            dilated_masks=np.packbits(masks), canvas4_delta=delta.astype(np.int16), psnr=psnr,
                            ssim=ssim, metrics_txt=np.array(rec["metrics_txt"]), clip_sha256=np.array(clips),
                            l_t=np.array(l_ts), hole_counts=np.array([len(v) for v in holes]),
                            hole_u8=np.concatenate(holes), schedule=np.array(repr(rec["schedule"])))
        print(name, "done:", rec["metrics_txt"].splitlines()[-1])


def _replay_net(replay, masks):
    """A stand-in network returning, for the i-th window, values that quantise to the recorded uint8 output at every
    hole pixel of the local frames (and 0 elsewhere, which the composite does not read)."""
    import hashlib
    import numpy as np
    import torch
    calls = []

    def net(x, l_t):
        i = len(calls)
        calls.append(i)
        sha, want_l_t, u8 = replay[i]
        assert hashlib.sha256(x.numpy().tobytes()).hexdigest() == sha and l_t == want_l_t
        pred = torch.from_numpy((u8.astype(np.float32) + 0.5) / 255 * 2 - 1).permute(0, 3, 1, 2)
        out = torch.zeros(x.shape[1:], dtype=torch.float32)
        out[:l_t] = pred
        return out, None
    return net


if __name__ == "__main__":
    main(sys.argv[1:])
