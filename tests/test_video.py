"""Video-level driver (SURVEY §8(f) rank 4): oracle vs the UNMODIFIED test.py's output, host logic on CPU (kernels
replaced by the oracle, tests only), 2-rank window sharding over gloo, and — on the GPU — the four byte-exact kernels
and the whole driver against the goldens."""
import ast
import hashlib
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from e2fgvi_b200 import video as V
from e2fgvi_b200.synth import synth_state_dict, synth_video
from oracle import restate, restate_video as RV

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# must equal oracle/gen_golden_video.py:CASES  (name -> model, n, H, W, family, weight seed, video seed, driver kwargs)
CASES = {
    "video_hq_tiny": ("e2fgvi_hq", 12, 100, 200, "stress", 0, 11, {}),
    "video_hq_numref": ("e2fgvi_hq", 23, 60, 108, "stress", 1, 12, dict(num_ref=2, ref_length=4, neighbor_stride=3)),
}


def _case(name):
    model, n, h, w, family, wseed, vseed, kw = CASES[name]
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    frames, raw = synth_video(n, h, w, vseed)
    masks = np.stack([RV.dilate_cross(m) for m in raw])
    return model, family, wseed, frames, masks, kw, g


@pytest.mark.parametrize("name", sorted(CASES))
def test_schedule_and_mask_dilation_match_test_py(name):
    model, family, wseed, frames, masks, kw, g = _case(name)
    n, h, w = masks.shape
    assert np.array_equal(np.unpackbits(g["dilated_masks"])[:n * h * w].reshape(n, h, w), masks)
    want = ast.literal_eval(str(g["schedule"]))
    assert [tuple(x) for x in want] == RV.window_schedule(n, **kw) == V.window_schedule(n, **kw)


def test_get_ref_index_properties():
    for length in (1, 7, 23, 61):
        for stride, step, num_ref in ((5, 10, -1), (3, 4, 2), (5, 10, 4), (2, 3, 1)):
            a = V.window_schedule(length, stride, step, num_ref)
            assert a == RV.window_schedule(length, stride, step, num_ref)
            covered = set()
            for f, nb, ref in a:
                assert not set(nb) & set(ref) and f in nb
                covered |= set(nb)
            assert covered == set(range(length))
    assert V.padded_size(100, 200) == (120, 216) and V.padded_size(240, 432) == (240, 432)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_driver_vs_reference_test_py(name):
    """restate_video + the oracle network reproduce what the unmodified test.py wrote: identical up to the <= 4e-6
    difference between the oracle network and the reference network, which can flip a uint8 truncation by 1 LSB."""
    model, family, wseed, frames, masks, kw, g = _case(name)
    mine = importlib.import_module("e2fgvi_b200.model." + model).InpaintGenerator()
    sd = synth_state_dict(mine, family, wseed)
    comp = RV.finalize(RV.inpaint_video(lambda x, l: restate.inpaint_generator_forward(sd, x, l), frames, masks, **kw))
    d = np.abs(comp.astype(np.int32) - g["comp"].astype(np.int32))
    assert d.max() <= 1 and (d > 0).mean() < 1e-4


def test_oracle_driver_bit_exact_with_reference_network():
    """restate_video fed the reference network's own output reproduces test.py's frames bit for bit.  The output is
    replayed from ``video_hq_numref_refnet.npz`` (oracle/gen_golden_video.py): each window's clip must hash to the
    one the reference network was given, and its output comes back as values that quantise to the reference's
    uint8 at the hole pixels of the local frames, the only pixels of it the composite reads (test.py:167-174)."""
    model, family, wseed, frames, masks, kw, g = _case("video_hq_numref")
    r = np.load(os.path.join(GOLDEN, "video_hq_numref_refnet.npz"))
    sched = ast.literal_eval(str(g["schedule"]))
    ends = np.cumsum(r["hole_counts"])
    h, w = masks.shape[1:]
    calls = []

    def replay(x, l_t):
        i = len(calls)
        calls.append(i)
        assert hashlib.sha256(x.numpy().tobytes()).hexdigest() == r["clip_sha256"][i] and l_t == r["l_t"][i]
        p = np.zeros((l_t, h, w, 3), np.float32)
        p[masks[sched[i][1]].astype(bool)] = (r["hole_u8"][ends[i] - r["hole_counts"][i]:ends[i]] + 0.5) / 255 * 2 - 1
        pred = torch.zeros(x.shape[1:], dtype=torch.float32)
        pred[:l_t, :, :h, :w] = torch.from_numpy(p).permute(0, 3, 1, 2)
        return pred, None

    comp = RV.finalize(RV.inpaint_video(replay, frames, masks, **kw))
    assert len(calls) == len(r["l_t"])
    assert np.array_equal(comp, g["comp"])


class _ToyModel(torch.nn.Module):
    """Per-clip independent stand-in for InpaintGenerator with outputs in (-1, 1)."""

    def forward(self, x, l_t):
        b, t, c, h, w = x.shape
        y = torch.tanh(x.roll(1, 3) * 0.7 + x.mean(dim=(1, 2), keepdim=True) + 0.1 * l_t)
        return y.reshape(b * t, c, h, w), None


def _oracle_kernels(monkeypatch):
    monkeypatch.setattr(V, "prepare_clip", lambda f, m, ids, hp, wp: RV.prepare_clip(f, m, ids, hp, wp))

    def compose(pred, frames, masks, ids, n_local, out=None):
        img = RV.compose(pred, frames, masks, ids, n_local)
        return img if out is None else out.copy_(img)
    monkeypatch.setattr(V, "compose", compose)
    monkeypatch.setattr(V, "blend", RV.blend)
    monkeypatch.setattr(V, "finalize", RV.finalize_canvas)


@pytest.mark.parametrize("clips_per_call", [1, 3])
def test_driver_host_logic_cpu(monkeypatch, clips_per_call):
    """Window grouping / batching / ordered blend of VideoInpainter == the sequential reference loop, exactly."""
    _oracle_kernels(monkeypatch)
    frames, raw = synth_video(32, 50, 70, 5)
    masks = np.stack([RV.dilate_cross(m) for m in raw])
    toy = _ToyModel()
    for kw in ({}, dict(num_ref=2, ref_length=4, neighbor_stride=3)):
        want = RV.finalize(RV.inpaint_video(lambda x, l: toy(x, l), frames, masks, **kw))
        got = V.VideoInpainter(toy, clips_per_call=clips_per_call, **kw)(torch.from_numpy(frames), torch.from_numpy(masks),
                                                                        device="cpu")
        assert np.array_equal(got.numpy(), want)


def test_driver_rejects_bad_inputs():
    # the reference indexes imgs[:, ref_ids] with an id == video_length here (IndexError at test.py:152); so do we
    bad = V.VideoInpainter(_ToyModel(), num_ref=2, ref_length=4, neighbor_stride=3)
    with pytest.raises(IndexError):
        bad(torch.zeros(31, 8, 8, 3, dtype=torch.uint8), torch.zeros(31, 8, 8, dtype=torch.uint8), device="cpu")
    with pytest.raises(IndexError):
        RV.inpaint_video(_ToyModel(), np.zeros((31, 8, 8, 3), np.uint8), np.zeros((31, 8, 8), np.uint8), 3, 4, 2)
    v = V.VideoInpainter(_ToyModel())
    with pytest.raises(TypeError):
        v(torch.zeros(4, 8, 8, 3), torch.zeros(4, 8, 8, dtype=torch.uint8), device="cpu")
    with pytest.raises(ValueError):
        v(torch.zeros(4, 8, 8, 3, dtype=torch.uint8), torch.zeros(4, 8, 9, dtype=torch.uint8), device="cpu")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        v(torch.zeros(4, 8, 8, 3, dtype=torch.uint8), torch.zeros(4, 8, 8, dtype=torch.uint8), device="cpu")


def _dist_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import pytest as _pytest
    from e2fgvi_b200 import clips as C
    r, w, _ = C.init_from_env("gloo")
    mp_ = _pytest.MonkeyPatch()
    _oracle_kernels(mp_)
    frames, raw = synth_video(23, 40, 60, 7)
    masks = np.stack([RV.dilate_cross(m) for m in raw])
    toy = _ToyModel()
    want = RV.finalize(RV.inpaint_video(lambda x, l: toy(x, l), frames, masks))
    got = V.VideoInpainter(toy, clips_per_call=2, rank=r, world=w)(torch.from_numpy(frames), torch.from_numpy(masks),
                                                                   device="cpu")
    q.put((rank, bool(np.array_equal(got.numpy(), want))))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    mp_.undo()


def test_two_rank_window_sharding_gloo():
    """Windows dealt round-robin to 2 ranks, uint8 all-gather, ordered blend on every rank == the sequential loop."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, 29631, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok in res)


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_video_kernels_bit_exact(cuda):
    frames, raw = synth_video(9, 50, 70, 3)
    masks = np.stack([RV.dilate_cross(m) for m in raw])
    f_cpu, m_cpu = torch.from_numpy(frames), torch.from_numpy(masks)
    f, m = f_cpu.to(cuda), m_cpu.to(cuda)
    ids = [7, 0, 3, 8, 2]
    ids_d = torch.tensor(ids, dtype=torch.int32, device=cuda)
    hp, wp = V.padded_size(50, 70)
    got = V.prepare_clip(f, m, ids_d, hp, wp)
    want = RV.prepare_clip(f_cpu, m_cpu, ids, hp, wp)
    assert torch.equal(got.cpu().view(torch.int32), want.view(torch.int32))          # bit pattern, incl. -0.0
    g = torch.Generator().manual_seed(0)
    pred = torch.tanh(torch.randn(5, 3, hp, wp, generator=g) * 2)
    pred[0, :, :4, :4] = 1.0                                                           # saturated tanh -> 255
    pred[1, :, :4, :4] = -1.0
    img = V.compose(pred.to(cuda), f, m, ids_d, 3)
    want_img = RV.compose(pred, f_cpu, m_cpu, ids, 3)
    assert torch.equal(img.cpu(), want_img)
    comp = torch.full((9, 50, 70, 3), -7.0, device=cuda)
    comp_ref = comp.cpu().clone()
    for first in ([1, 1, 1], [0, 1, 0], [0, 0, 0]):
        fd = torch.tensor(first, dtype=torch.int32, device=cuda)
        V.blend(img, ids_d[:3], fd, comp)
        RV.blend(want_img, ids[:3], first, comp_ref)
        img = img.flip(0).contiguous()
        want_img = want_img.flip(0).contiguous()
    assert torch.equal(comp.cpu()[[7, 0, 3]], comp_ref[[7, 0, 3]])
    assert torch.equal(V.finalize(comp[[7, 0, 3]].contiguous()).cpu(), RV.finalize_canvas(comp_ref[[7, 0, 3]]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_video_driver_vs_reference_test_py(cuda, name):
    """The whole driver on the GPU against what the unmodified test.py wrote.  The network's output differs from the
    reference's by <= ~2e-4 (fp16 DCN / attention operands), i.e. <= 0.03 LSB before the uint8 truncation, so a few
    percent of the hole pixels may land on the neighbouring integer; everything outside the holes is exact."""
    model, family, wseed, frames, masks, kw, g = _case(name)
    net = importlib.import_module("model." + model)
    gen = net.InpaintGenerator().eval()
    gen.load_state_dict(synth_state_dict(gen, family, wseed), strict=True)
    gen.to(cuda)
    for cpc in (1, 4):
        got = V.VideoInpainter(gen, clips_per_call=cpc, **kw)(torch.from_numpy(frames), torch.from_numpy(masks)).cpu().numpy()
        d = np.abs(got.astype(np.int32) - g["comp"].astype(np.int32))
        hole = masks.astype(bool)
        assert d[~hole].max() == 0
        assert d.max() <= 1 and (d[hole] > 0).mean() < 0.05, (d.max(), (d[hole] > 0).mean())
