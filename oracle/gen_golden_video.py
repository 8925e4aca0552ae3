"""TEST INFRASTRUCTURE — runs the UNMODIFIED ``/root/reference/test.py`` (its ``main_worker``) on a synthetic video
in the build container and stores what it wrote, as the golden for the video-level driver (SURVEY §8(f) rank 4).

    python -m oracle.gen_golden_video        # only where /root/reference exists

How the script is made to run offline without touching it: ``matplotlib`` (not installed; only used for the final
preview window) is replaced by ``unittest.mock`` modules, ``mmcv`` comes from ``oracle/mmcv_shim``, frames / masks /
checkpoint are written to a temp dir as PNGs and a ``torch.save``d synthetic ``state_dict``, and ``cv2.VideoWriter``
is replaced by a recorder so the composited frames are captured losslessly instead of being mp4-encoded.
Inputs are NOT stored: ``e2fgvi_b200.synth.synth_video`` / ``synth_state_dict`` regenerate them from seeds.
"""
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")

# name -> (model, n_frames, H, W, family, weight seed, video seed, extra test.py argv)
CASES = {
    "video_hq_tiny": ("e2fgvi_hq", 12, 100, 200, "stress", 0, 11, []),
    "video_hq_numref": ("e2fgvi_hq", 23, 60, 108, "stress", 1, 12, ["--num_ref", "2", "--step", "4",
                                                                   "--neighbor_stride", "3"]),
}

CHILD = r'''
import sys, os, runpy, types
from unittest import mock
import numpy as np
shim, ref, tmp, out = sys.argv[1:5]
argv = sys.argv[5:]
sys.path[:] = [shim, ref] + [p for p in sys.path if p not in ("", os.getcwd())]
for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation", "matplotlib.patches", "matplotlib.path"):
    sys.modules[name] = mock.MagicMock(name=name)
import cv2
written = []
class Recorder:
    def __init__(self, *a, **k): pass
    def write(self, bgr): written.append(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB).copy())   # undo the script's swap
    def release(self): pass
cv2.VideoWriter = Recorder
os.chdir(tmp)                       # the script writes ./results/
sys.argv = [os.path.join(ref, "test.py")] + argv
glb = runpy.run_path(os.path.join(ref, "test.py"), run_name="__main__")
# the dilated masks the script used, and its schedule helper on a few probes
masks = glb["read_mask"](argv[argv.index("-m") + 1], written[0].shape[1::-1])
masks = np.stack([(np.array(m) != 0).astype(np.uint8) for m in masks])
sched = []
n = len(written)
stride = glb["neighbor_stride"]
for f in range(0, n, stride):
    nb = [i for i in range(max(0, f - stride), min(n, f + stride + 1))]
    sched.append((f, nb, glb["get_ref_index"](f, nb, n)))
np.savez_compressed(out, comp=np.stack(written), dilated_masks=np.packbits(masks),
                    schedule=np.array(repr(sched)))
print("captured", len(written), "frames", written[0].shape)
'''


def main():
    import cv2
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import importlib
    from e2fgvi_b200.synth import synth_state_dict, synth_video
    from oracle.reference_loader import REFERENCE_ROOT, SHIM
    os.makedirs(OUT, exist_ok=True)
    for name, (model, n, h, w, family, wseed, vseed, extra) in CASES.items():
        frames, masks = synth_video(n, h, w, vseed)
        with tempfile.TemporaryDirectory() as tmp:
            os.makedirs(os.path.join(tmp, "frames"))
            os.makedirs(os.path.join(tmp, "masks"))
            for i in range(n):
                cv2.imwrite(os.path.join(tmp, "frames", f"{i:05d}.png"), cv2.cvtColor(frames[i], cv2.COLOR_RGB2BGR))
                cv2.imwrite(os.path.join(tmp, "masks", f"{i:05d}.png"), masks[i] * 255)
            mine = importlib.import_module("e2fgvi_b200.model." + model).InpaintGenerator()
            torch.save(synth_state_dict(mine, family, wseed), os.path.join(tmp, "ckpt.pth"))
            child = os.path.join(tmp, "child.py")
            with open(child, "w") as f:
                f.write(CHILD)
            argv = ["-v", os.path.join(tmp, "frames"), "-c", os.path.join(tmp, "ckpt.pth"), "-m",
                    os.path.join(tmp, "masks"), "--model", model] + extra
            subprocess.check_call([sys.executable, child, SHIM, REFERENCE_ROOT, tmp, os.path.join(OUT, name + ".npz")]
                                  + argv, cwd=tmp)
        print(name, "done")
    gen_network_replay()


def gen_network_replay(name="video_hq_numref"):
    """The reference NETWORK driven by ``oracle/restate_video.py`` on one case, for
    ``tests/test_video.py::test_oracle_driver_bit_exact_with_reference_network``.  Written only when that run equals
    what test.py wrote, bit for bit.  The network's output reaches the composite only as the uint8 value of each hole
    pixel of the window's local frames (test.py:167-174), so that is what is kept, with a SHA-256 of every clip the
    network was given."""
    import hashlib
    import importlib
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    from e2fgvi_b200.synth import synth_state_dict, synth_video
    from oracle import restate_video as RV
    from oracle.reference_loader import reference_generator
    model, n, h, w, family, wseed, vseed, extra = CASES[name]
    kw = dict(num_ref=int(extra[extra.index("--num_ref") + 1]), ref_length=int(extra[extra.index("--step") + 1]),
              neighbor_stride=int(extra[extra.index("--neighbor_stride") + 1]))
    frames, raw = synth_video(n, h, w, vseed)
    masks = np.stack([RV.dilate_cross(m) for m in raw])
    ref = reference_generator(hq=model == "e2fgvi_hq")
    ref.load_state_dict(synth_state_dict(importlib.import_module("e2fgvi_b200.model." + model).InpaintGenerator(),
                                         family, wseed), strict=True)
    clips, l_ts, holes = [], [], []
    sched = RV.window_schedule(n, **kw)

    def net(x, l_t):
        i = len(clips)
        clips.append(hashlib.sha256(x.numpy().tobytes()).hexdigest())
        l_ts.append(l_t)
        pred, flows = ref(x, l_t)
        p = (((pred[:l_t, :, :h, :w] + 1) / 2).permute(0, 2, 3, 1).numpy() * 255).astype(np.uint8)
        holes.append(p[masks[sched[i][1]].astype(bool)])
        return pred, flows

    comp = RV.finalize(RV.inpaint_video(net, frames, masks, **kw))
    assert np.array_equal(comp, np.load(os.path.join(OUT, name + ".npz"))["comp"]), "driver != test.py"
    np.savez_compressed(os.path.join(OUT, name + "_refnet.npz"), clip_sha256=np.array(clips), l_t=np.array(l_ts),
                        hole_counts=np.array([len(v) for v in holes]), hole_u8=np.concatenate(holes))
    print(name + "_refnet", len(clips), "windows", sum(len(v) for v in holes), "hole pixels")


if __name__ == "__main__":
    if "--network-replay-only" in sys.argv:
        gen_network_replay()
    else:
        main()
