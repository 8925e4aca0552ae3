"""Dataset evaluation (``e2fgvi_b200.evaluate``) against what the UNMODIFIED evaluate.py computed
(``tests/golden/eval_*.npz``, written by ``oracle/gen_golden_eval.py``): the loader, the window schedule, the oracle
driver and metrics (CPU), the evaluator's host logic with the kernels replaced by the oracle on one rank and on two
gloo ranks (CPU), and on the GPU the canvas, the metrics and the command line."""
import ast
import hashlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from e2fgvi_b200 import evaluate as E
from e2fgvi_b200 import video as V
from e2fgvi_b200.synth import synth_state_dict, write_eval_dataset
from oracle import restate_metrics as RM
from oracle import restate_video as RV

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# must equal oracle/gen_golden_eval.py:CASES  (name -> model, weight family, weight seed, dataset seed, videos)
CASES = {
    "eval_e2fgvi": ("e2fgvi", "stress", 3, 21, [("bear", 11), ("car-turn", 7)]),
    "eval_hq": ("e2fgvi_hq", "stress", 4, 22, [("swan", 16)]),
}


def golden_case(name, tmp):
    """Regenerate the case's dataset under ``tmp`` and load it -> (frames, masks, evaluate.py's canvas, golden)."""
    model, family, wseed, dseed, videos = CASES[name]
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    write_eval_dataset(str(tmp), videos, seed=dseed)
    loaded = [E.load_test_video(str(tmp), "davis", v) for v, _ in videos]
    frames = np.concatenate([f for f, _ in loaded])
    masks = np.concatenate([m for _, m in loaded])
    canvas = ((frames.astype(np.int32) * 4 + g["canvas4_delta"]) / 4).astype(np.float32)
    return frames, masks, canvas, g


def _video_lines(txt):
    return txt.splitlines()[:-1]


def _final_numbers(line):
    return [float(x) for x in re.search(r"SSIM[^:]*: ([\d.]+)/([\d.]+)", line).groups()]


@pytest.mark.parametrize("name", sorted(CASES))
def test_loader_matches_reference_test_dataset(name, tmp_path):
    """load_test_video on the generator's dataset == what the reference TestDataset loaded, byte for byte."""
    model, family, wseed, dseed, videos = CASES[name]
    frames, masks, canvas, g = golden_case(name, tmp_path)
    start = 0
    for (v, n), sha in zip(videos, g["frames_sha256"]):
        assert hashlib.sha256(frames[start:start + n].tobytes()).hexdigest() == sha
        start += n
    assert np.array_equal(np.unpackbits(g["dilated_masks"])[:masks.size].reshape(masks.shape), masks)
    assert list(g["names"]) == [v for v, _ in videos] and E.video_names(str(tmp_path), "davis") == dict(videos)


def test_evaluate_py_schedule_is_num_ref_minus_one():
    table = ast.literal_eval(str(np.load(os.path.join(GOLDEN, "eval_e2fgvi.npz"))["schedule"]))
    assert sorted(table) == list(range(1, 61))
    for n, windows in table.items():
        assert [tuple(x) for x in windows] == V.window_schedule(n, num_ref=-1) == RV.window_schedule(n)


def _replay_model(g, masks, offsets):
    """Stands in for the network: each clip is identified by its SHA-256 among the windows evaluate.py ran, and gets
    back values that quantise to the network's uint8 output at its local frames' hole pixels."""
    shas = list(g["clip_sha256"])
    ends = np.cumsum(g["hole_counts"])

    class Replay(torch.nn.Module):
        def forward(self, x, l_t):
            outs = []
            for clip in x:
                sha = hashlib.sha256(clip.unsqueeze(0).numpy().tobytes()).hexdigest()
                i = shas.index(sha)
                assert l_t == g["l_t"][i]
                nb = offsets[i]
                p = np.zeros((l_t,) + masks.shape[1:] + (3,), np.float32)
                p[masks[nb].astype(bool)] = (g["hole_u8"][ends[i] - g["hole_counts"][i]:ends[i]] + 0.5) / 255 * 2 - 1
                pred = torch.zeros(clip.shape, dtype=torch.float32)
                pred[:l_t] = torch.from_numpy(p).permute(0, 3, 1, 2)
                outs.append(pred)
            return torch.cat(outs), None
    return Replay()


def _window_frames(name):
    """Global (concatenated) local frame ids of every window, in evaluate.py's order."""
    out, start = [], 0
    for _, n in CASES[name][4]:
        out += [[start + i for i in nb] for _, nb, _ in RV.window_schedule(n)]
        start += n
    return out


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_driver_and_metrics_reproduce_evaluate_py(name, tmp_path):
    """restate_video fed the reference network's output reproduces evaluate.py's canvas bit for bit, and the oracle
    metrics its per-frame values and its metrics-file lines."""
    frames, masks, canvas, g = golden_case(name, tmp_path)
    net = _replay_model(g, masks, _window_frames(name))
    start, lines = 0, []
    for k, (v, n) in enumerate(CASES[name][4]):
        sl = slice(start, start + n)
        comp = np.stack([c.astype(np.float32) for c in RV.inpaint_video(net, frames[sl], masks[sl])])
        assert np.array_equal(comp, canvas[sl])
        pr = [RM.calc_psnr_and_ssim(a, b) for a, b in zip(frames[sl], comp)]
        assert [p for p, _ in pr] == list(g["psnr"][sl]) and [s for _, s in pr] == list(g["ssim"][sl])
        lines.append(E.video_line(k, len(CASES[name][4]), v, [p for p, _ in pr], [s for _, s in pr]))
        start += n
    txt = str(g["metrics_txt"])
    assert lines == _video_lines(txt)
    assert _final_numbers(E.summary_line(list(g["psnr"]), list(g["ssim"]))) == _final_numbers(txt.splitlines()[-1])


def _oracle_kernels(mp):
    mp.setattr(V, "prepare_clip", lambda f, m, ids, hp, wp: RV.prepare_clip(f, m, ids, hp, wp))

    def compose(pred, frames, masks, ids, n_local, out=None):
        img = RV.compose(pred, frames, masks, ids, n_local)
        return img if out is None else out.copy_(img)
    mp.setattr(V, "compose", compose)
    mp.setattr(V, "blend", RV.blend)
    mp.setattr(V, "finalize", RV.finalize_canvas)

    def psnr_ssim(ref, test):
        p, s = zip(*[RM.calc_psnr_and_ssim(a, b) for a, b in zip(ref.numpy(), test.numpy())])
        return torch.tensor(p, dtype=torch.float64), torch.tensor(s, dtype=torch.float64)
    mp.setattr(E.metrics, "psnr_ssim", psnr_ssim)


def _run_host(name, data, out_dir, rank=0, world=1, save=False):
    frames, masks, canvas, g = golden_case(name, data)
    printed = []
    res = E.evaluate_dataset(_replay_model(g, masks, _window_frames(name)), str(data), "davis", str(out_dir),
                             "m.txt", save_results=save, num_workers=0, device="cpu", rank=rank, world=world,
                             out=printed.append)
    return printed, res, g, canvas


def test_evaluator_host_logic_cpu(monkeypatch, tmp_path):
    """evaluate_dataset with the kernels replaced by the oracle writes evaluate.py's lines, byte for byte, and the
    uint8 canvases with --save_results."""
    _oracle_kernels(monkeypatch)
    out = tmp_path / "out"
    out.mkdir()
    printed, res, g, canvas = _run_host("eval_e2fgvi", tmp_path / "data", out, save=True)
    txt = str(g["metrics_txt"])
    assert printed[:-1] == _video_lines(txt)
    assert _final_numbers(printed[-1]) == _final_numbers(txt.splitlines()[-1])
    assert printed[-1].startswith("Finish evaluation... Average Frame PSNR/SSIM: ")
    assert (out / "m.txt").read_text() == "\n".join(printed)
    assert res["bear"][0] + res["car-turn"][0] == list(g["psnr"])
    import cv2
    png = cv2.cvtColor(cv2.imread(str(out / "car-turn" / "00003.png")), cv2.COLOR_BGR2RGB)
    assert np.array_equal(png, canvas[11 + 3].astype(np.uint8))


def _dist_worker(rank, world, port, tmp, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import pytest as _pytest
    from e2fgvi_b200 import clips as C
    C.init_from_env("gloo")
    mp_ = _pytest.MonkeyPatch()
    _oracle_kernels(mp_)
    out = os.path.join(tmp, "out")
    os.makedirs(out, exist_ok=True)
    printed, res, g, _ = _run_host("eval_e2fgvi", os.path.join(tmp, f"data{rank}"), out, rank, world)
    q.put((rank, printed, sorted(res)))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    mp_.undo()


def test_two_rank_video_sharding_gloo(monkeypatch, tmp_path):
    """Videos dealt to 2 ranks: rank 0 prints and writes exactly what one rank does."""
    import torch.multiprocessing as mp
    _oracle_kernels(monkeypatch)
    (tmp_path / "one").mkdir()
    single, _, _, _ = _run_host("eval_e2fgvi", tmp_path / "data", tmp_path / "one")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, 29641, str(tmp_path), q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict((r, (printed, names)) for r, printed, names in [q.get(timeout=300) for _ in procs])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][0] == single and res[1][0] == []
    assert res[0][1] == ["bear", "car-turn"] and res[1][1] == ["car-turn"]
    assert (tmp_path / "out" / "m.txt").read_text() == (tmp_path / "one" / "m.txt").read_text()


# ------------------------------------------------------------------------------------------------------------- GPU
def _generator(name, cuda):
    import importlib
    model, family, wseed, _, _ = CASES[name]
    gen = importlib.import_module("e2fgvi_b200.model." + model).InpaintGenerator().eval()
    gen.load_state_dict(synth_state_dict(gen, family, wseed), strict=True)
    return gen.to(cuda)


@pytest.mark.gpu
def test_composite_then_finalize_is_call(cuda):
    from e2fgvi_b200.synth import synth_video
    frames, raw = synth_video(12, 60, 108, 4)
    masks = torch.from_numpy(np.stack([RV.dilate_cross(m) for m in raw]))
    vi = V.VideoInpainter(_generator("eval_hq", cuda))
    comp = vi.composite(torch.from_numpy(frames), masks)
    assert comp.dtype == torch.float32 and comp.is_cuda and comp.shape == (12, 60, 108, 3)
    assert torch.equal(V.finalize(comp), vi(torch.from_numpy(frames), masks))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_evaluate_video_vs_evaluate_py(cuda, name, tmp_path):
    """The network differs from the reference's by <= ~2e-4, which can flip a uint8 truncation inside the holes;
    everything outside them is exact, and the metrics of our canvas equal the oracle's metrics of it."""
    frames, masks, canvas, g = golden_case(name, tmp_path)
    vi = V.VideoInpainter(_generator(name, cuda))
    start = 0
    for v, n in CASES[name][4]:
        sl = slice(start, start + n)
        p, s, comp = E.evaluate_video(vi, torch.from_numpy(frames[sl]), torch.from_numpy(masks[sl]))
        comp = comp.cpu().numpy()
        hole = np.repeat(masks[sl].astype(bool)[..., None], 3, axis=3)
        d = np.abs(comp - canvas[sl])
        assert d[~hole].max() == 0 and d.max() <= 1.0
        p, s = p.cpu().numpy(), s.cpu().numpy()
        assert np.abs(p - g["psnr"][sl]).max() <= 0.01 and np.abs(s - g["ssim"][sl]).max() <= 1e-4
        op, os_ = zip(*[RM.calc_psnr_and_ssim(a, b) for a, b in zip(frames[sl], comp)])
        assert np.abs(p - np.array(op)).max() <= 1e-9 and np.abs(s - np.array(os_)).max() <= 1e-9
        start += n


@pytest.mark.gpu
def test_command_line(cuda, tmp_path):
    """``python -m e2fgvi_b200.evaluate`` on the golden dataset: evaluate.py's lines, within the network tolerance."""
    name = "eval_e2fgvi"
    model, family, wseed, dseed, videos = CASES[name]
    write_eval_dataset(str(tmp_path / "data"), videos, seed=dseed)
    import importlib
    gen = importlib.import_module("e2fgvi_b200.model." + model).InpaintGenerator()
    torch.save(synth_state_dict(gen, family, wseed), str(tmp_path / "ckpt.pth"))
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "e2fgvi_b200.evaluate", "--dataset", "davis", "--data_root",
                        str(tmp_path / "data"), "--model", model, "--ckpt", str(tmp_path / "ckpt.pth"), "--num_workers",
                        "2"], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    txt = (tmp_path / "results" / f"{model}_davis" / f"{model}_davis_metrics.txt").read_text()
    assert txt.splitlines()[-1] in r.stdout
    want = str(np.load(os.path.join(GOLDEN, name + ".npz"))["metrics_txt"]).splitlines()
    got = txt.splitlines()
    assert len(got) == len(want)
    for a, b in zip(got[:-1], want[:-1]):
        assert a.split("|")[0] == b.split("|")[0]
        pa, sa = map(float, a.split(": ")[-1].split("/"))
        pb, sb = map(float, b.split(": ")[-1].split("/"))
        assert abs(pa - pb) <= 0.01 and abs(sa - sb) <= 1e-4
    assert np.allclose(_final_numbers(got[-1]), _final_numbers(want[-1]), atol=0.011)
