"""Video-level driver — the host-side mirror of the reference's ``test.py`` inference loop (SURVEY §8(f) rank 4).

Reference: ``test.py:37-52`` (``get_ref_index``), ``:146-151`` (sliding-window schedule), ``:152-166`` (mask, mirror pad,
forward), ``:167-179`` (crop, uint8, hole composite, 0.5/0.5 blend), ``:195`` (final uint8).  Same names and argument
meaning (``neighbor_stride``, ``ref_length`` = ``--step``, ``num_ref``); the per-window tensor work runs as four
byte-exact CUDA kernels on uint8 frames resident in HBM (``csrc/video.cu``) instead of eager torch + numpy on the host,
so a video makes ONE host->device trip (uint8) and one trip back (uint8).

Windows are independent units of work (only the final blend is ordered), so

* windows with the same shape ``(len(neighbor_ids), len(ref_ids))`` are batched into one ``InpaintGenerator.forward``;
* with ``world > 1`` windows are dealt round-robin to ranks, each rank composes its windows' uint8 frames, one
  ``all_gather`` exchanges them (uint8: 4x smaller than the fp32 predictions, SURVEY §8(e)), and every rank blends in
  schedule order.

There is no CPU path: the kernels raise on CPU tensors.
"""
import torch

from . import _lib
from .ops import _need_cuda, _stream

MOD_H, MOD_W = 60, 108          # test.py:157-158


def get_ref_index(f, neighbor_ids, length, ref_length=10, num_ref=-1):
    """Non-local reference frame ids of the window centred on ``f`` (test.py:37-52; ``ref_length`` / ``num_ref`` are
    module globals there).  ``num_ref == -1``: every ``ref_length``-th frame of the whole video outside the window;
    otherwise frames ``f +- ref_length * (num_ref // 2)`` (the reference's ``>`` test admits ``num_ref + 1`` of them)."""
    neighbors = set(neighbor_ids)
    if num_ref == -1:
        return [i for i in range(0, length, ref_length) if i not in neighbors]
    start = max(0, f - ref_length * (num_ref // 2))
    end = min(length, f + ref_length * (num_ref // 2))
    out = []
    for i in range(start, end + 1, ref_length):
        if i not in neighbors:
            if len(out) > num_ref:
                break
            out.append(i)
    return out


def window_schedule(video_length, neighbor_stride=5, ref_length=10, num_ref=-1):
    """``[(f, neighbor_ids, ref_ids)]`` in the order the reference visits them (test.py:146-151)."""
    out = []
    for f in range(0, video_length, neighbor_stride):
        nb = list(range(max(0, f - neighbor_stride), min(video_length, f + neighbor_stride + 1)))
        out.append((f, nb, get_ref_index(f, nb, video_length, ref_length, num_ref)))
    return out


def padded_size(h, w):
    """Model input size after mirror padding to multiples of (60, 108) (test.py:157-160)."""
    return h + (MOD_H - h % MOD_H) % MOD_H, w + (MOD_W - w % MOD_W) % MOD_W


# ----------------------------------------------------------------------------------------------- kernel wrappers
def prepare_clip(frames, masks, ids, hp, wp):
    """uint8 frames (N,H,W,3) + masks (N,H,W) + int32 ids (t,) -> masked, normalised, mirror-padded (t,3,hp,wp) fp32."""
    _need_cuda(frames, masks, ids)
    n, h, w, _ = frames.shape
    t = ids.numel()
    out = torch.empty((t, 3, hp, wp), dtype=torch.float32, device=frames.device)
    st = _lib.load().e2f_video_prepare_clip(frames.data_ptr(), masks.data_ptr(), ids.data_ptr(), out.data_ptr(), t, h, w,
                                            hp, wp, _stream())
    _lib.check(st, "e2f_video_prepare_clip")
    return out


def compose(pred, frames, masks, ids, n_local, out=None):
    """pred (>=n_local,3,hp,wp) fp32 -> img (n_local,H,W,3) uint8: hole pixels from the prediction, the rest original."""
    _need_cuda(pred, frames, masks, ids)
    n, h, w, _ = frames.shape
    hp, wp = pred.shape[-2:]
    if out is None:
        out = torch.empty((n_local, h, w, 3), dtype=torch.uint8, device=frames.device)
    pred = pred.contiguous()
    st = _lib.load().e2f_video_compose(pred.data_ptr(), frames.data_ptr(), masks.data_ptr(), ids.data_ptr(),
                                       out.data_ptr(), n_local, h, w, hp, wp, _stream())
    _lib.check(st, "e2f_video_compose")
    return out


def blend(img, ids, first, comp):
    """comp[ids[k]] = first[k] ? img[k] : 0.5*comp + 0.5*img[k]  (in place, fp32)."""
    _need_cuda(img, ids, first, comp)
    n_local = ids.numel()
    st = _lib.load().e2f_video_blend(img.data_ptr(), ids.data_ptr(), first.data_ptr(), comp.data_ptr(), n_local,
                                     comp[0].numel(), _stream())
    _lib.check(st, "e2f_video_blend")
    return comp


def finalize(comp):
    _need_cuda(comp)
    out = torch.empty(comp.shape, dtype=torch.uint8, device=comp.device)
    st = _lib.load().e2f_video_finalize(comp.data_ptr(), out.data_ptr(), comp.numel(), _stream())
    _lib.check(st, "e2f_video_finalize")
    return out


# ----------------------------------------------------------------------------------------------- the driver
class VideoInpainter:
    """``VideoInpainter(model)(frames_u8, masks_u8) -> comp_u8`` == the loop of test.py:146-195 around
    ``model(masked_imgs, len(neighbor_ids))``.

    frames (N,H,W,3) uint8 RGB and masks (N,H,W) uint8 (non-zero = hole, already dilated) may live on the host (they
    are uploaded once) or on the GPU.  ``clips_per_call`` same-shape windows share one forward."""

    def __init__(self, model, neighbor_stride=5, ref_length=10, num_ref=-1, clips_per_call=4, rank=0, world=1,
                 cuda_graphs=True):
        self.model = model
        # every window shape (clips per call, local frames, reference frames) repeats across a video and across
        # videos: replay a CUDA graph per shape instead of ~200 Python-side launches per forward
        if cuda_graphs and hasattr(model, "enable_cuda_graphs") and getattr(model, "_graphs", None) is None:
            model.enable_cuda_graphs(True, max_shapes=8)
        self.neighbor_stride, self.ref_length, self.num_ref = neighbor_stride, ref_length, num_ref
        self.clips_per_call = max(1, clips_per_call)
        self.rank, self.world = rank, world

    def schedule(self, video_length):
        """The window list; raises IndexError where the reference's ``imgs[:1, neighbor_ids + ref_ids]`` (test.py:152)
        would: with ``num_ref != -1`` its ``range(start, end_idx + 1, ...)`` can emit the id ``video_length`` itself."""
        sched = window_schedule(video_length, self.neighbor_stride, self.ref_length, self.num_ref)
        for f, _, ref in sched:
            if any(i >= video_length for i in ref):
                raise IndexError(f"index {max(ref)} is out of bounds for the {video_length}-frame video (window f={f}; "
                                 "test.py:45-46 lets get_ref_index reach video_length when num_ref != -1)")
        return sched

    @torch.no_grad()
    def __call__(self, frames, masks, device=None):
        """-> (N,H,W,3) uint8 on the device: the frames test.py writes (test.py:195)."""
        return finalize(self.composite(frames, masks, device))

    @torch.no_grad()
    def composite(self, frames, masks, device=None):
        """-> (N,H,W,3) fp32 on the device: the blended canvas before the final uint8 truncation, which is what
        evaluate.py scores (evaluate.py:113-114,125-126)."""
        device = torch.device(device) if device is not None else (
            frames.device if frames.is_cuda else torch.device("cuda", torch.cuda.current_device()))
        if frames.dtype != torch.uint8 or masks.dtype != torch.uint8:
            raise TypeError("frames and masks must be uint8 (frames RGB in [0,255], masks non-zero = hole)")
        if frames.dim() != 4 or frames.shape[-1] != 3 or masks.shape != frames.shape[:3]:
            raise ValueError(f"frames must be (N,H,W,3) and masks (N,H,W); got {tuple(frames.shape)} / {tuple(masks.shape)}")
        frames = frames.to(device, non_blocking=True).contiguous()
        masks = masks.to(device, non_blocking=True).contiguous()
        n, h, w, _ = frames.shape
        hp, wp = padded_size(h, w)
        sched = self.schedule(n)
        mine = [wi for wi in range(len(sched)) if wi % self.world == self.rank]
        max_local = max(len(nb) for _, nb, _ in sched)
        share = (len(sched) + self.world - 1) // self.world
        # this rank's composed windows, padded to (share, max_local) so that the all-gather is rectangular
        imgs = torch.zeros((share, max_local, h, w, 3), dtype=torch.uint8, device=device)
        ids_dev = {wi: torch.tensor(sched[wi][1] + sched[wi][2], dtype=torch.int32, device=device) for wi in mine}
        # same-shape windows -> one forward
        groups = {}
        for wi in mine:
            groups.setdefault((len(sched[wi][1]), len(sched[wi][2])), []).append(wi)
        for (n_local, _), wis in groups.items():
            for i in range(0, len(wis), self.clips_per_call):
                batch = wis[i:i + self.clips_per_call]
                clips = torch.stack([prepare_clip(frames, masks, ids_dev[wi], hp, wp) for wi in batch])
                pred, _ = self.model(clips, n_local)
                t = clips.shape[1]
                pred = pred.view(len(batch), t, 3, hp, wp)
                for j, wi in enumerate(batch):
                    compose(pred[j], frames, masks, ids_dev[wi], n_local, out=imgs[wi // self.world, :n_local])
        if self.world > 1:
            import torch.distributed as dist
            gathered = torch.empty((self.world,) + tuple(imgs.shape), dtype=torch.uint8, device=device)
            dist.all_gather_into_tensor(gathered.view(-1, *imgs.shape[1:]), imgs)
        else:
            gathered = imgs.unsqueeze(0)
        # ordered blend (test.py:175-179): window wi lives at gathered[wi % world, wi // world]
        comp = torch.empty((n, h, w, 3), dtype=torch.float32, device=device)
        seen = [False] * n
        for wi, (_, nb, _) in enumerate(sched):
            first = torch.tensor([0 if seen[i] else 1 for i in nb], dtype=torch.int32, device=device)
            nb_dev = torch.tensor(nb, dtype=torch.int32, device=device)
            blend(gathered[wi % self.world, wi // self.world, :len(nb)], nb_dev, first, comp)
            for i in nb:
                seen[i] = True
        assert all(seen), "every frame is a neighbour of some window (test.py:147-150)"
        return comp
