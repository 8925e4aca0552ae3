"""Dataset evaluation — the B200 counterpart of the reference's ``evaluate.py``: inpaint every video of DAVIS or
YouTube-VOS at 432x240 and report per-frame PSNR / SSIM averaged per video and over the dataset.

    python -m e2fgvi_b200.evaluate --dataset davis --data_root datasets --model e2fgvi_hq --ckpt release_model/E2FGVI-HQ-CVPR22.pth
    python -m torch.distributed.run --nproc-per-node 8 -m e2fgvi_b200.evaluate ...     # videos sharded over 8 GPUs

Reference: ``evaluate.py:70-162`` (window loop, composite, blend, metrics, summary lines), ``core/dataset.py:82-135``
(``TestDataset``), ``core/utils.py:59-84`` (``TestZipReader``).  The window loop with ``num_ref = -1`` is
``VideoInpainter.composite`` (the fp32 canvas the reference scores, ``evaluate.py:113-114``), and the metrics are one
``e2f_psnr_ssim`` call per video (``metrics.psnr_ssim``); a video's frames, canvas and metrics stay on the GPU and only
2·N doubles come back.  Loading (zip member order, cv2 decode, PIL resize, NEAREST mask resize, ``> 0``, 3x3 cross
dilation x4) runs on the host in DataLoader workers, so video i+1 loads while video i is on the GPU.

With ``world > 1`` rank r evaluates videos r, r+world, ... whole; rank 0 gathers the per-frame values and writes the
lines in dataset order, identical to a single rank's output.  VFID is not computed: it needs the I3D network and
weights the reference does not ship.
"""
import argparse
import importlib
import json
import os
import sys
import zipfile

import numpy as np
import torch

from . import metrics, video

SIZE = (432, 240)                  # (w, h), evaluate.py:17


def _dilate(m):
    import cv2
    return cv2.dilate(m, cv2.getStructuringElement(cv2.MORPH_CROSS, (3, 3)), iterations=4)


def video_names(data_root, dataset):
    """``{name: frame_count}`` of ``<data_root>/<dataset>/test.json`` in file order (core/dataset.py:86-90)."""
    with open(os.path.join(data_root, dataset, "test.json")) as f:
        return json.load(f)


def load_test_video(data_root, dataset, name, size=SIZE, length=None):
    """One video as ``TestDataset.load_item`` reads it -> ``(frames (N,H,W,3) uint8 RGB, masks (N,H,W) uint8 0/1)``.

    Frame ``idx`` is member ``sorted(namelist())[idx]`` of ``JPEGImages/<name>.zip`` decoded by cv2 and resized by PIL
    with its default filter; the mask is ``test_masks/<name>/%05d.png`` resized NEAREST, converted to L, ``> 0`` and
    dilated with a 3x3 cross 4 times.  ``length`` defaults to the count in ``test.json``."""
    import cv2
    from PIL import Image
    if length is None:
        length = video_names(data_root, dataset)[name]
    root = os.path.join(data_root, dataset)
    frames, masks = [], []
    with zipfile.ZipFile(os.path.join(root, "JPEGImages", f"{name}.zip")) as z:
        members = sorted(z.namelist())
        for idx in range(length):
            bgr = cv2.imdecode(np.frombuffer(z.read(members[idx]), np.uint8), cv2.IMREAD_COLOR)
            img = Image.fromarray(cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB)).convert("RGB").resize(size)
            frames.append(np.asarray(img, dtype=np.uint8))
            mask = Image.open(os.path.join(root, "test_masks", name, f"{idx:05d}.png")).resize(size, Image.NEAREST)
            masks.append(_dilate((np.asarray(mask.convert("L")) > 0).astype(np.uint8)))
    return np.stack(frames), np.stack(masks)


class _Videos(torch.utils.data.Dataset):
    def __init__(self, data_root, dataset, names, size):
        self.data_root, self.dataset, self.names, self.size = data_root, dataset, names, size

    def __len__(self):
        return len(self.names)

    def __getitem__(self, i):
        name, length = self.names[i]
        frames, masks = load_test_video(self.data_root, self.dataset, name, self.size, length)
        return torch.from_numpy(frames), torch.from_numpy(masks), name


@torch.no_grad()
def evaluate_video(inpainter, frames_u8, masks_u8, device=None):
    """-> ``(psnr (N,) fp64, ssim (N,) fp64, comp (N,H,W,3) fp32)`` on the device: evaluate.py:82-126 for one video,
    the canvas scored against the original frames."""
    device = torch.device(device) if device is not None else (
        frames_u8.device if frames_u8.is_cuda else torch.device("cuda", torch.cuda.current_device()))
    frames = frames_u8.to(device, non_blocking=True).contiguous()
    comp = inpainter.composite(frames, masks_u8, device)
    psnr, ssim = metrics.psnr_ssim(frames, comp)
    return psnr, ssim, comp


def video_line(index, count, name, psnr, ssim):
    """evaluate.py:133-138; ``name`` is shown as the DataLoader collated it, a 1-tuple."""
    cur_psnr = sum(psnr) / len(psnr)
    cur_ssim = sum(ssim) / len(ssim)
    return f'[{index + 1:3}/{count}] Name: {str((name,)):25} | PSNR/SSIM: {cur_psnr:.4f}/{cur_ssim:.4f}'


def summary_line(all_psnr, all_ssim):
    """evaluate.py:155-160 without VFID."""
    return ('Finish evaluation... Average Frame PSNR/SSIM: '
            f'{sum(all_psnr) / len(all_psnr):.2f}/{sum(all_ssim) / len(all_ssim):.4f}')


def evaluate_dataset(model, data_root, dataset, result_path, summary_name, save_results=False, num_workers=4,
                     device=None, rank=0, world=1, size=SIZE, out=print):
    """Evaluate every video of ``<data_root>/<dataset>/test.json`` with ``model``; rank 0 writes
    ``<result_path>/<summary_name>`` and prints the same lines through ``out``.  Returns ``{name: (psnr list,
    ssim list)}`` for all videos on rank 0 and for this rank's videos elsewhere."""
    names = list(video_names(data_root, dataset).items())
    mine = list(range(rank, len(names), world))
    loader = torch.utils.data.DataLoader(_Videos(data_root, dataset, [names[i] for i in mine], size), batch_size=None,
                                         shuffle=False, num_workers=num_workers)
    inpainter = video.VideoInpainter(model, world=1)
    summary = open(os.path.join(result_path, summary_name), "w") if rank == 0 else None
    results = {}

    def emit(i, name):
        line = video_line(i, len(names), name, *results[name])
        out(line)
        summary.write(line + "\n")

    for k, (frames, masks, name) in enumerate(loader):
        psnr, ssim, comp = evaluate_video(inpainter, frames, masks, device)
        results[name] = (psnr.cpu().tolist(), ssim.cpu().tolist())
        if world == 1:
            emit(mine[k], name)
        if save_results:                                              # evaluate.py:142-151
            import cv2
            path = os.path.join(result_path, name)
            os.makedirs(path, exist_ok=False)
            for i, frame in enumerate(video.finalize(comp).cpu().numpy()):
                cv2.imwrite(os.path.join(path, str(i).zfill(5) + ".png"), cv2.cvtColor(frame, cv2.COLOR_RGB2BGR))
    if world > 1:
        import torch.distributed as dist
        parts = [None] * world
        dist.all_gather_object(parts, results)
        if rank == 0:
            for part in parts:
                results.update(part)
            for i, (name, _) in enumerate(names):
                emit(i, name)
    if rank == 0:
        all_psnr = [v for name, _ in names for v in results[name][0]]
        all_ssim = [v for name, _ in names for v in results[name][1]]
        line = summary_line(all_psnr, all_ssim)
        out(line)
        summary.write(line)
        summary.close()
    return results


def main(argv=None):
    parser = argparse.ArgumentParser(description="E2FGVI evaluation (PSNR / SSIM) on the B200")
    parser.add_argument("--dataset", choices=["davis", "youtube-vos"], type=str, required=True)
    parser.add_argument("--data_root", type=str, required=True)
    parser.add_argument("--model", choices=["e2fgvi", "e2fgvi_hq"], type=str, required=True)
    parser.add_argument("--ckpt", type=str, required=True)
    parser.add_argument("--save_results", action="store_true", default=False)
    parser.add_argument("--num_workers", default=4, type=int)
    args = parser.parse_args(argv)

    from .clips import init_from_env
    rank, world, local_rank = init_from_env()
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    net = importlib.import_module("e2fgvi_b200.model." + args.model)
    model = net.InpaintGenerator().to(device)
    model.load_state_dict(torch.load(args.ckpt, map_location=device), strict=True)
    model.eval()
    if rank == 0:
        print(f"Loading from: {args.ckpt}")
        print("Start evaluation...")
    result_path = os.path.join("results", f"{args.model}_{args.dataset}")
    os.makedirs(result_path, exist_ok=True)
    evaluate_dataset(model, args.data_root, args.dataset, result_path, f"{args.model}_{args.dataset}_metrics.txt",
                     save_results=args.save_results, num_workers=args.num_workers, device=device, rank=rank,
                     world=world)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    sys.exit(main())
