"""Drop-in for the reference's `src.evaluate` (/root/reference/src/evaluate.py): same CLI flags, same
`evaluate_on_test(opt, checkpoint_model_path, output_dir, save_images)` entry point and the same final line
`Test AUCs - SSIM(best ws=..): .., MSE: .., PSNR: ..` -- but batched and on the GPU end to end:

  reference (src/evaluate.py:204-265)                    here
  ----------------------------------------------------   ---------------------------------------------------
  batch_size forced to 1, one D2H copy per image          images run in batches (--batch-size, default 64)
  SR -> uint8 via 5 tiny kernels + numpy                  truncation fused into the SR model's last kernel
  ssim_numpy Python loop, 14 calls per image (~12 s)      ONE scoring launch per batch: all window sizes + MSE + PSNR
  roc_auc_score on the host                               unchanged (N_img scalars), after an all_gather when sharded

Deviation (documented in DESIGN.md): the model runs with evaluation semantics (DropPath off); the reference
never calls model.eval() on this path, which makes its AUC nondeterministic (SURVEY.md section 0, item 2).
With --workers / torchrun the images shard by index across ranks and only the [n_img, n_ws+2] score
table is gathered (NCCL), as SURVEY.md section 8e prescribes.
"""
from __future__ import annotations

import argparse
import glob
import os
import re
import sys
from pathlib import Path
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import metrics, ops
from .main import DRCT as DRCTOpt
from .main import DRN as DRNOpt
from .main import setup_opt_drct, setup_opt_drn


# ------------------------------------------------------------------------------------------ CLI (src/evaluate.py:20-45)
def parse_args(argv=None):
    pre = argparse.ArgumentParser(add_help=False)
    pre.add_argument('--config', type=str, default=None)
    pre_args, _ = pre.parse_known_args(argv)
    p = argparse.ArgumentParser(description='Evaluation entrypoint', parents=[pre])
    p.add_argument('--model-type', type=str, default='drct', choices=['drct', 'drn-l'])
    p.add_argument('--dataset', type=str, default='mvtec', choices=['mvtec'])
    p.add_argument('--classe', type=str, default='grid')
    p.add_argument('--scale', type=int, default=4)
    p.add_argument('--resolution', type=int, default=128)
    p.add_argument('--device', type=str, default='auto', choices=['auto', 'cuda', 'mps', 'cpu'])
    p.add_argument('--data-root', type=str, default='auto')
    p.add_argument('--run-dir', type=str, default='')
    p.add_argument('--checkpoint', type=str, default='')
    p.add_argument('--batch-size', type=int, default=64)
    p.add_argument('--output-dir', type=str, default='')
    p.add_argument('--save-images', action='store_true', default=True)
    p.add_argument('--workers', type=int, default=0 if sys.platform == 'darwin' else 4)
    # localisation: per-pixel anomaly maps (1 - SSIM of one window size, squared error), their max as image scores, pixel AUROC
    p.add_argument('--anomaly-maps', action='store_true', default=False,
                   help='also compute per-pixel 1-SSIM and squared-error maps and report the AUCs of their per-image max')
    p.add_argument('--map-window-size', type=int, default=11, help='SSIM window size of the 1-SSIM map (odd)')
    p.add_argument('--map-sigma', type=float, default=4.0, help='Gaussian smoothing of both maps (scipy gaussian_filter sigma; 0 = off)')
    p.add_argument('--gms-map', action='store_true', default=False,
                   help='also compute the multi-scale gradient-magnitude-similarity (MSGMS) map, smoothed with --map-sigma, and report '
                        'every map metric for it too; implies --anomaly-maps')
    p.add_argument('--mask-dir', type=str, default=None,
                   help='ground-truth masks <mask-dir>/<stem>.png or <stem>_mask.png (non-zero = defect): adds pixel AUROC; '
                        'implies --anomaly-maps')
    p.add_argument('--save-maps', action='store_true', default=False,
                   help='write <output-dir>/maps/<split>/<stem>_ssim.npy and <stem>_se.npy (float32 HxW; also <stem>_gms.npy with '
                        '--gms-map); implies --anomaly-maps')
    p.add_argument('--au-pro', type=float, nargs='?', const=0.3, default=None, metavar='FPR_LIMIT',
                   help='also report the AU-PRO of both maps up to this false-positive rate (bare flag: 0.3); needs --mask-dir')
    p.add_argument('--pr-metrics', action='store_true', default=False,
                   help='also report the pixel AP and the F1-max of both maps with the threshold that attains it; needs --mask-dir')
    p.add_argument('--save-segmentation', action='store_true', default=False,
                   help='write <output-dir>/segmentation/<split>/<stem>_{ssim,se[,gms]}.png: each map thresholded at its F1-max threshold '
                        '(uint8 0 / 255); needs --mask-dir, implies --pr-metrics')
    # thresholds calibrated on defect-free images: no test label is used to choose them
    p.add_argument('--calibration-dir', type=str, default=None,
                   help='defect-free images laid out like a test split (HR/ and an LR folder, e.g. <data-root>/<classe>/train/good): '
                        'a pixel and an image threshold per map are calibrated on them and the test set is scored at them; implies '
                        '--anomaly-maps')
    p.add_argument('--calibration-quantile', type=float, default=0.999, metavar='Q',
                   help='the thresholds are this quantile (in (0, 1]) of the calibration pixels and of the calibration images\' map maxima; '
                        'a pixel / image is defective when its score is above it')
    p.add_argument('--save-calibrated-masks', action='store_true', default=False,
                   help='write <output-dir>/calibrated/<split>/<stem>_{ssim,se[,gms]}.png: each map thresholded at its calibrated pixel '
                        'threshold (uint8 0 / 255); needs --calibration-dir')
    if pre_args.config and os.path.isfile(pre_args.config):
        import yaml

        with open(pre_args.config, 'r') as f:
            cfg = yaml.safe_load(f) or {}
        p.set_defaults(**{k.replace('-', '_'): v for k, v in cfg.items()})
    args = p.parse_args(argv)
    if args.au_pro is not None:
        if args.mask_dir is None:
            p.error('--au-pro needs --mask-dir (the ground-truth masks define the defect regions)')
        if not 0.0 < args.au_pro <= 1.0:
            p.error(f'--au-pro: the false-positive-rate limit must be in (0, 1], got {args.au_pro}')
    if (args.pr_metrics or args.save_segmentation) and args.mask_dir is None:
        p.error('--pr-metrics and --save-segmentation need --mask-dir (the ground-truth masks label the defect pixels)')
    if not 0.0 < args.calibration_quantile <= 1.0:
        p.error(f'--calibration-quantile must be in (0, 1], got {args.calibration_quantile}')
    if args.save_calibrated_masks and args.calibration_dir is None:
        p.error('--save-calibrated-masks needs --calibration-dir (the defect-free images the threshold is calibrated on)')
    return args


def infer_from_run_dir(run_dir: str):
    """src/evaluate.py:48-122: path-name pattern first, then config.txt overrides."""
    result = {'model_type': None, 'dataset': None, 'classe': None, 'resolution': None, 'scale': None}
    for seg in Path(run_dir).parts:
        if seg in ('drct', 'drn-l'):
            result['model_type'] = seg
            break
    m = re.match(r"(?P<ds>\w+)_(?P<cls>\w+)_(?P<res>\d+)_X(?P<scale>\d+)", Path(run_dir).name)
    if m:
        result['dataset'], result['classe'] = m.group('ds'), m.group('cls')
        result['resolution'], result['scale'] = int(m.group('res')), int(m.group('scale'))
    cfg_path = Path(run_dir) / 'config.txt'
    if cfg_path.exists():
        try:
            lines = cfg_path.read_text().splitlines()

            def read_val(key):
                for line in lines:
                    if line.strip().startswith(f"{key}:"):
                        return line.split(':', 1)[1].strip()
                return None

            for key, field in (('model_name', 'model_type'), ('dataset', 'dataset'), ('classe', 'classe')):
                v = read_val(key)
                if v:
                    result[field] = v
            res = read_val('patch_size')
            if res and res.isdigit():
                result['resolution'] = int(res)
            scale_val = read_val('upscale') or read_val('scale')
            if scale_val:
                ms = re.findall(r"\d+", scale_val)
                if ms:
                    result['scale'] = int(ms[-1])
        except Exception:
            pass
    return result


def resolve_checkpoint(args):
    if args.checkpoint:
        return args.checkpoint
    if args.run_dir:
        for name in ('model_best.pt', 'model_latest.pt'):
            cand = os.path.join(args.run_dir, 'model', name)
            if os.path.isfile(cand):
                return cand
    raise FileNotFoundError('Please provide --checkpoint or a valid --run-dir containing model/*.pt')


# ------------------------------------------------------------------------------------------ data (src/data.py, test mode)
def _rgb_to_y(img: np.ndarray) -> np.ndarray:
    """skimage.color.rgb2ycbcr(img)[..., 0] for uint8 RGB (used by src/data.py:59 when n_colors == 1)."""
    f = img.astype(np.float64) / 255.0
    return 16.0 + 65.481 * f[..., 0] + 128.553 * f[..., 1] + 24.966 * f[..., 2]


def _set_channel(img: np.ndarray, n_colors: int) -> np.ndarray:
    if img.ndim == 2:
        img = img[:, :, None]
    c = img.shape[2]
    if n_colors == 1 and c == 3:
        img = _rgb_to_y(img)[:, :, None]
    elif n_colors == 3 and c == 1:
        img = np.concatenate([img] * 3, 2)
    return img


def scan_split(data_dir: str, scale: int) -> Tuple[List[str], List[str]]:
    """HR/*.png sorted + matching LR file, same candidate order as src/data.py:109-134."""
    names_hr = sorted(glob.glob(os.path.join(data_dir, 'HR', '*.png')))
    names_lr = []
    for f in names_hr:
        stem = os.path.splitext(os.path.basename(f))[0]
        cands = [os.path.join(data_dir, 'LR_bicubic', f'X{scale}', f'{stem}x{scale}.png'),
                 os.path.join(data_dir, f'LR_{scale}', f'{stem}.png'), os.path.join(data_dir, 'LR', f'{stem}.png')]
        for c in cands:
            if os.path.exists(c):
                names_lr.append(c)
                break
        else:
            raise FileNotFoundError(f"LR image not found for {stem} at scale {scale}: tried {', '.join(cands)}")
    return names_hr, names_lr


def load_pair(f_hr: str, f_lr: str, scale: int, n_colors: int, rgb_range: float, raw_u8: bool = False):
    """-> (lr [nc,h,w] float32, hr [nc,H,W] float32) in [0, rgb_range] (src/data.py:11-19, 84-92, 176-183).
    raw_u8: when both decoded images are uint8 and rgb_range == 255 (the reference default: the float conversion and the evaluator's
    uint8 truncation are then exact inverses) return the uint8 HWC arrays instead -- a quarter of the bytes cross PCIe and the float
    scaling runs on the device (adsr_u8_to_float_nchw); same results."""
    from PIL import Image

    hr = _set_channel(np.array(Image.open(f_hr)), n_colors)
    lr = _set_channel(np.array(Image.open(f_lr)), n_colors)
    ih, iw = lr.shape[:2]
    hr = hr[0:ih * scale, 0:iw * scale]
    if raw_u8 and hr.dtype == np.uint8 and lr.dtype == np.uint8 and float(rgb_range) == 255.0:
        return torch.from_numpy(np.ascontiguousarray(lr)), torch.from_numpy(np.ascontiguousarray(hr))
    to_t = lambda a: torch.from_numpy(np.ascontiguousarray(a.transpose(2, 0, 1))).float().mul_(rgb_range / 255)
    return to_t(lr), to_t(hr)


# ------------------------------------------------------------------------------------------ batched device path
class BatchedEvaluator:
    """SR forward + uint8 truncation + per-image scores for batches of (lr, hr) pairs.

    `step(lr, hr)` takes what the reference's loader yields (float tensors in [0, rgb_range], on the host or
    already on the device) and returns the fp64 score table [B, n_ws + 2] on the device; nothing else leaves
    the GPU.  Host tensors are copied with non_blocking=True (pin them for overlap).

    maps = (win_size, sigma) also computes the anomaly maps of every step (ops.anomaly_maps on the step's uint8 SR / HR):
    `last_maps` = (1 - SSIM map, squared-error map, per-image max of both), next to `last_sr_u8` and `last_hr_u8`.  gms=True (needs maps)
    adds the MSGMS map of the same sigma (ops.gms_map): `last_maps` = (1 - SSIM map, squared-error map, MSGMS map, per-image max of the
    three [B, 3]).  Either way the maps are all entries but the last, the maxima the last one."""

    def __init__(self, model, rgb_range: float, window_sizes: Optional[Sequence[int]] = None,
                 maps: Optional[Tuple[int, float]] = None, gms: bool = False):
        if gms and maps is None:
            raise ValueError("gms=True needs maps=(win_size, sigma): the MSGMS map comes with the other maps and uses their sigma")
        self.model = model
        self.rgb_range = float(rgb_range)
        self.window_sizes = list(window_sizes) if window_sizes is not None else None
        self.maps = (int(maps[0]), float(maps[1])) if maps is not None else None
        self.gms = bool(gms)
        self.device = torch.device('cuda')
        self.last_sr_u8: Optional[torch.Tensor] = None
        self.last_hr_u8: Optional[torch.Tensor] = None
        self.last_maps: Optional[Tuple[torch.Tensor, ...]] = None
        self._copy_stream = None
        self._graphs = {}
        self.use_graph = os.environ.get('ADSR_CUDA_GRAPH', '1') != '0'
        self._bufs = [None, None]
        self._next_buf = 0
        self._host_ring = [None, None, None]
        self._host_next = 0

    def step(self, lr: torch.Tensor, hr: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        lr_d = lr.to(self.device, non_blocking=True)
        hr_d = hr.to(self.device, non_blocking=True)
        if lr.is_cuda and hr.is_cuda and out is None:         # device-resident inputs: the step can be replayed as a CUDA graph
            return self._score_graphed(lr_d, hr_d)
        return self._score(lr_d, hr_d, out)

    # ---- the whole step (~1000 kernel launches through the C ABI) as ONE CUDA graph per static input buffer pair
    def _score_graphed(self, lr_d: torch.Tensor, hr_d: torch.Tensor) -> torch.Tensor:
        """First call for a buffer pair runs eagerly (workspaces, packed weights), the second one is captured, later ones
        replay the graph.  The returned table (and last_sr_u8, last_hr_u8, last_maps) are the graph's static outputs: valid until
        the next replay."""
        if not self.use_graph or ops.PROFILE is not None:
            return self._score(lr_d, hr_d)
        target = self.model.model if hasattr(self.model, 'model') else self.model
        packed = target._pack() if hasattr(target, '_pack') else None     # repacked weights (new parameters) -> a new graph
        key = (lr_d.data_ptr(), hr_d.data_ptr(), tuple(lr_d.shape), tuple(hr_d.shape), lr_d.dtype, hr_d.dtype,
               tuple(self.window_sizes) if self.window_sizes is not None else None, id(packed), self.maps, self.gms)
        ent = self._graphs.get(key)
        if ent is None:
            while len(self._graphs) >= 8:                     # evict the oldest entry only (no recapture thrash)
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = {"graph": None, "keep": (lr_d, hr_d, packed)}
            return self._score(lr_d, hr_d)
        if ent["graph"] is None:
            try:
                torch.cuda.synchronize(self.device)
                n0 = ops.LAUNCHES
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    ent["out"] = self._score(lr_d, hr_d)
                    ent["sr_u8"] = self.last_sr_u8
                    ent["hr_u8"] = self.last_hr_u8
                    ent["maps"] = self.last_maps
                ent["launches"] = ops.LAUNCHES - n0
                ops.LAUNCHES = n0
                ent["graph"] = g
                # the graph holds raw addresses of the model's workspaces: keep them alive for as long as the graph is, even
                # if the model's own workspace cache evicts them
                ent["ws"] = dict(getattr(target, '_ws_cache', {}))
            except Exception as e:                            # capture not possible: stay on the eager path (still no fallback
                self.use_graph = False                        # away from the CUDA kernels)
                print(f"[adsr] CUDA graph capture disabled: {e}", file=sys.stderr)
                return self._score(lr_d, hr_d)
        ent["graph"].replay()
        ops.LAUNCHES += ent["launches"]
        self.last_sr_u8 = ent["sr_u8"]
        self.last_hr_u8 = ent["hr_u8"]
        self.last_maps = ent["maps"]
        return ent["out"]

    def _score(self, lr_d: torch.Tensor, hr_d: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if hr_d.dtype == torch.uint8:                         # already quantised NHWC
            hr_u8 = hr_d
        else:
            hr_u8 = ops.quantize_u8(hr_d, self.rgb_range)
        h, w = hr_u8.shape[1], hr_u8.shape[2]
        target = self.model.model if hasattr(self.model, 'model') else self.model
        if lr_d.dtype == torch.uint8:                         # decoded PNG bytes: np2Tensor (src/data.py:11-17) on the device
            lr_d = ops.u8_to_float(lr_d, self.rgb_range)
        _, sr_u8 = target.run(lr_d, want_float=False, want_u8=True)
        if sr_u8.shape[1] != h or sr_u8.shape[2] != w:        # sr = sr[..., :h, :w]  (src/evaluate.py:212-213)
            sr_u8 = sr_u8[:, :h, :w, :].contiguous()
        if self.window_sizes is None:
            self.window_sizes = metrics.window_sizes_for(min(h, w))
        self.last_sr_u8 = sr_u8
        self.last_hr_u8 = hr_u8
        scores = metrics.score_batch(sr_u8, hr_u8, self.window_sizes, out)
        self.last_maps = ops.anomaly_maps(sr_u8, hr_u8, *self.maps) if self.maps is not None else None
        if self.gms:
            gms, gms_max = ops.gms_map(sr_u8, hr_u8, self.maps[1])
            self.last_maps = self.last_maps[:2] + (gms, torch.cat([self.last_maps[2], gms_max[:, None]], 1))
        return scores

    # ---- double-buffered input path: the host -> device copies of batch i + 1 run on a copy stream while batch i is computed
    def submit(self, lr: torch.Tensor, hr: torch.Tensor):
        """Start the (pinned) host -> device copies of one batch on the copy stream; returns a handle for step_submitted().
        Two persistent device buffer sets alternate (no allocation per batch): at most one submitted batch may be pending
        while another one is being computed."""
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        k = self._next_buf
        self._next_buf ^= 1
        key = (tuple(lr.shape), lr.dtype, tuple(hr.shape), hr.dtype)
        buf = self._bufs[k]
        if buf is None or buf[0] != key:
            buf = [key, torch.empty(lr.shape, dtype=lr.dtype, device=self.device), torch.empty(hr.shape, dtype=hr.dtype, device=self.device),
                   None]                                       # [key, lr_d, hr_d, event: the compute that last read this set]
            self._bufs[k] = buf
            # fresh blocks may be memory the caching allocator just took back from kernels still pending on the compute
            # stream (per-call temporaries, the previous sr_u8): the copies below must not overtake them
            self._copy_stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self._copy_stream):
            if buf[3] is not None:
                self._copy_stream.wait_event(buf[3])           # the batch computed from this buffer set two submits ago is done
            buf[1].copy_(lr, non_blocking=True)
            buf[2].copy_(hr, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self._copy_stream)
        return k, done

    def step_submitted(self, handle, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        k, done = handle
        buf = self._bufs[k]
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(done)
        scores = self._score_graphed(buf[1], buf[2]) if out is None else self._score(buf[1], buf[2], out)
        buf[3] = torch.cuda.Event()
        buf[3].record(cur)
        return scores

    def to_host_async(self, t: torch.Tensor):
        """Starts the device -> host read of a (small) result tensor into a pinned ring buffer and returns (host tensor, event):
        the caller enqueues the NEXT step first and only then `event.synchronize()`s -- the GPU never idles while the host turns
        a step around.  The host tensor is valid until three more reads have been started."""
        k = self._host_next
        self._host_next = (k + 1) % len(self._host_ring)
        buf = self._host_ring[k]
        if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
            buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            self._host_ring[k] = buf
        buf.copy_(t, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        return buf, ev

    def run_pipelined(self, batches):
        """Iterates (lr, hr) host batches with one batch of copy look-ahead; yields the device score table of each batch
        (a private copy: the CUDA graph's static output tensor is overwritten by the next replay of the same buffer set)."""
        it = iter(batches)
        try:
            nxt = self.submit(*next(it))
        except StopIteration:
            return
        while nxt is not None:
            cur = nxt
            try:
                nxt = self.submit(*next(it))
            except StopIteration:
                nxt = None
            yield self.step_submitted(cur).clone()


def _dist_info():
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def gather_scores(local_scores: torch.Tensor, local_ids: torch.Tensor, n_total: int, to_host: bool = True):
    """ONE all_gather (NCCL over NVLink when sharded) of the per-rank score rows with the image id as an extra fp64 column
    (ids < 2^53 are exact); <= 8*(n_ws+3) bytes per image: latency only (SURVEY.md section 8e).
    to_host=True: rank 0 returns the numpy table ordered by image id, other ranks None.
    to_host=False: every rank returns the gathered DEVICE tensor [world * n_max, C + 1] (pad rows carry id -1) without any
    host synchronisation; pass it to `scores_table` when the table is consumed."""
    import torch.distributed as dist

    rank, world = _dist_info()
    c = local_scores.shape[1]
    n = local_scores.shape[0]
    n_max = n if world == 1 else (n_total + world - 1) // world
    packed = local_scores.new_full((n_max, c + 1), -1.0)
    packed[:n, :c] = local_scores
    packed[:n, c] = local_ids.to(local_scores.dtype)
    if world == 1:
        gathered = packed
    else:
        gathered = packed.new_empty((world * n_max, c + 1))
        dist.all_gather_into_tensor(gathered, packed)
    if not to_host:
        return gathered
    return scores_table(gathered, n_total) if rank == 0 else None


def scores_table(gathered: torch.Tensor, n_total: int) -> np.ndarray:
    """Gathered device rows (gather_scores(..., to_host=False)) -> host table [n_total, C] ordered by image id."""
    arr = gathered.cpu().numpy()
    c = arr.shape[1] - 1
    keep = arr[:, c] >= 0
    out = np.empty((n_total, c), dtype=np.float64)
    out[arr[keep, c].astype(np.int64)] = arr[keep, :c]
    return out


def find_mask(mask_dir: str, hr_path: str, label: int) -> Optional[str]:
    """Ground-truth mask of HR image `<stem>.png`: `<mask_dir>/<stem>.png`, else `<mask_dir>/<stem>_mask.png`; None for a good image
    without one (all clear).  A bad image needs a mask."""
    stem = os.path.splitext(os.path.basename(hr_path))[0]
    cands = [os.path.join(mask_dir, f'{stem}.png'), os.path.join(mask_dir, f'{stem}_mask.png')]
    for c in cands:
        if os.path.exists(c):
            return c
    if label:
        raise FileNotFoundError(f"mask not found for defective image {hr_path}: tried {', '.join(cands)}")
    return None


def load_mask(path: Optional[str], hr_shape: Tuple[int, int], crop: Tuple[int, int]) -> np.ndarray:
    """bool [H, W] defect mask (any non-zero channel), cropped like its HR image (`hr[0:crop[0], 0:crop[1]]`); None = all clear."""
    from PIL import Image

    if path is None:
        return np.zeros(hr_shape, dtype=bool)
    m = np.array(Image.open(path))
    m = (m != 0).any(axis=2) if m.ndim == 3 else m != 0
    m = m[0:crop[0], 0:crop[1]]
    if m.shape != tuple(hr_shape):
        raise ValueError(f"mask {path} is {m.shape[0]}x{m.shape[1]} after cropping, its image is {hr_shape[0]}x{hr_shape[1]}")
    return m


def hr_size(f_hr: str, f_lr: str, scale: int) -> Tuple[int, int]:
    """(H, W) of an HR image as load_pair crops it to its LR image, from the PNG headers."""
    from PIL import Image

    with Image.open(f_hr) as im_hr, Image.open(f_lr) as im_lr:
        return min(im_hr.size[1], im_lr.size[1] * scale), min(im_hr.size[0], im_lr.size[0] * scale)


def above(t: float) -> float:
    """The fp32 threshold of a strict decision: for every fp32 score x, x >= above(t) <=> x > t (t an fp32 value)."""
    return float(np.nextafter(np.float32(t), np.float32(np.inf)))


def save_sr_image(sr_u8_hwc: np.ndarray, output_dir: str, name: str, split: str, scale_value: int) -> None:
    from PIL import Image

    out_dir = Path(output_dir) / split / f"x{scale_value}"
    out_dir.mkdir(parents=True, exist_ok=True)
    img = Image.fromarray(sr_u8_hwc[:, :, 0] if sr_u8_hwc.shape[2] == 1 else sr_u8_hwc)
    img.save(str(out_dir / f"{name}.png"))


def evaluate_on_test(opt, checkpoint_model_path, output_dir: str, save_images: bool, batch_size: Optional[int] = None,
                     anomaly_maps: bool = False, map_window_size: int = 11, map_sigma: float = 4.0, mask_dir: Optional[str] = None,
                     save_maps: bool = False, au_pro: Optional[float] = None, pr_metrics: bool = False,
                     save_segmentation: bool = False, calibration_dir: Optional[str] = None, calibration_quantile: float = 0.999,
                     save_calibrated_masks: bool = False, gms_map: bool = False):
    """src/evaluate.py:138-267 with the loops batched.  Returns dict(best_ws, auc_ssim, auc_mse, auc_psnr, n, scores).

    anomaly_maps (implied by mask_dir / save_maps): per-pixel 1 - SSIM (window map_window_size) and squared-error maps, smoothed with
    a Gaussian of map_sigma; the AUCs of their per-image max are added as auc_map_ssim / auc_map_se (the maxima as `map_max`) and
    printed on a `Map AUCs - ...` line before the `Test AUCs - ...` line.  mask_dir adds the pixel-level AUROC of both maps
    (pixel_auroc_ssim / pixel_auroc_se; single process only), ranked on the device by metrics.LocalisationAccumulator.  au_pro (an FPR
    limit in (0, 1], needs mask_dir) adds the AU-PRO of both maps (au_pro_ssim / au_pro_se, pro_fpr_limit), printed on a `Map PRO - ...`
    line before the `Map AUCs - ...` line.  pr_metrics (needs mask_dir) adds the pixel AP and the F1-max of both maps with the score that
    attains it (pixel_ap_{ssim,se}, f1_max_{ssim,se}, f1_threshold_{ssim,se}), printed on a `Map PR - ...` line before the `Map PRO`
    line, or before the `Map AUCs` line without one.  The F1 threshold is an oracle threshold: picked with the ground truth it is scored
    on.  save_segmentation (needs mask_dir, implies pr_metrics) writes each map thresholded at its F1 threshold as a uint8 0 / 255 mask
    to <output_dir>/segmentation/<split>/<stem>_{ssim,se}.png.  save_maps writes <output_dir>/maps/<split>/<stem>_{ssim,se}.npy.

    calibration_dir (implies anomaly_maps; single process only): defect-free images in the layout of a test split, every one of a test
    image's HR size.  They run first; for each map the pixel threshold t_px is the calibration_quantile (in (0, 1], inverted_cdf: an
    actual score) of all their pixels and the image threshold t_img the same quantile of their map maxima.  Decisions are strict: a
    pixel is defective when map > t_px, an image when its map max > t_img, so at most a fraction 1 - q of the calibration pixels and
    images is flagged.  Adds calib_{pixel,image}_threshold_{ssim,se} and the test set's calib_image_{tpr,fpr}_{ssim,se}, with mask_dir
    also calib_pixel_{precision,recall,fpr,f1,iou,pro}_{ssim,se} at t_px, printed on a `Map CAL - ...` line before the other `Map`
    lines.  No test label is used to choose the thresholds.  save_calibrated_masks (needs calibration_dir) writes the `map > t_px` masks
    as uint8 0 / 255 to <output_dir>/calibrated/<split>/<stem>_{ssim,se}.png.

    gms_map (implies anomaly_maps) adds a third map kind, the multi-scale gradient-magnitude-similarity map smoothed with map_sigma:
    everything above is also computed for it, with the suffix _gms in the result keys and file names and `MSGMS` on the printed lines
    (after the SE entry of each kind)."""
    from .model import Model

    if au_pro is not None:
        if mask_dir is None:
            raise ValueError("au_pro needs mask_dir: the ground-truth masks define the defect regions")
        if not 0.0 < float(au_pro) <= 1.0:
            raise ValueError(f"au_pro: the false-positive-rate limit must be in (0, 1], got {au_pro}")
    if (pr_metrics or save_segmentation) and mask_dir is None:
        raise ValueError("pr_metrics and save_segmentation need mask_dir: the ground-truth masks label the defect pixels")
    if not 0.0 < float(calibration_quantile) <= 1.0:
        raise ValueError(f"calibration_quantile must be in (0, 1], got {calibration_quantile}")
    if save_calibrated_masks and calibration_dir is None:
        raise ValueError("save_calibrated_masks needs calibration_dir: the defect-free images the threshold is calibrated on")
    pr_metrics = pr_metrics or save_segmentation
    anomaly_maps = anomaly_maps or gms_map or mask_dir is not None or save_maps or calibration_dir is not None
    kinds = [('ssim', '1-SSIM'), ('se', 'SE')] + ([('gms', 'MSGMS')] if gms_map else [])   # (key / file suffix, printed label)
    n_maps = len(kinds)
    scale = opt.scale[-1] if isinstance(opt.scale, list) else int(opt.scale)
    rank, world = _dist_info()
    if mask_dir is not None and world > 1:
        raise RuntimeError("--mask-dir needs the whole maps of every image in one process: run it without sharding (world size 1)")
    if calibration_dir is not None and world > 1:
        raise RuntimeError("--calibration-dir needs the whole maps of every calibration image in one process: run it without sharding "
                           "(world size 1)")
    entries = []                                             # (label, split, hr path, lr path): good first, then bad
    for label, split in ((0, 'good'), (1, 'bad')):
        d = f'{opt.data_root}/{opt.classe}/test/{split}'
        hr_files, lr_files = scan_split(d, scale)
        entries += [(label, split, h, l) for h, l in zip(hr_files, lr_files)]
    y_true = [e[0] for e in entries]
    if len(set(y_true)) < 2:
        print('Test set lacks both classes; AUC not available')
        return None
    mask_paths = [find_mask(mask_dir, e[2], e[0]) for e in entries] if mask_dir is not None else None   # fail before the model runs

    # SSIM window sizes come from the smallest HR dimension over the WHOLE test set (src/evaluate.py:233-235), known from the
    # PNG headers before the images are sharded: every rank sweeps the same sizes, also one that holds no image at all
    from PIL import Image

    min_dim, test_sizes = None, set()
    for _, _, f_hr, f_lr in entries:
        dims = hr_size(f_hr, f_lr, scale)
        test_sizes.add(dims)
        min_dim = min(dims) if min_dim is None else min(min_dim, *dims)
    cal_files = []
    if calibration_dir is not None:                          # checked before the model runs
        cal_files = list(zip(*scan_split(calibration_dir, scale)))
        if not cal_files:
            raise ValueError(f"no calibration images in {calibration_dir}/HR")
        for f_hr, f_lr in cal_files:
            dims = hr_size(f_hr, f_lr, scale)
            if dims not in test_sizes:
                raise ValueError(f"calibration image {f_hr} is {dims[0]}x{dims[1]}, the test images are "
                                 f"{', '.join(f'{h}x{w}' for h, w in sorted(test_sizes))}")

    opt.pre_train = checkpoint_model_path
    model = Model(opt, None)
    ev = BatchedEvaluator(model, opt.rgb_range, metrics.window_sizes_for(min_dim),
                          maps=(map_window_size, map_sigma) if anomaly_maps else None, gms=gms_map)
    bs = batch_size or getattr(opt, 'eval_batch_size', None) or 64
    mine = list(range(rank, len(entries), world))            # image index i -> rank i mod R
    rows, ids = [], []

    def host_batches(files, ids_, order):
        """(lr, hr) pinned host batches of the (hr path, lr path) files[i] for i in ids_; `order` records the ids of each batch."""
        for s in range(0, len(ids_), bs):
            idx = ids_[s:s + bs]
            pairs = [load_pair(files[i][0], files[i][1], scale, opt.n_colors, opt.rgb_range, raw_u8=True) for i in idx]
            if len({p[0].dtype for p in pairs}) > 1:           # mixed decodes (should not happen within a dataset): all float
                pairs = [load_pair(files[i][0], files[i][1], scale, opt.n_colors, opt.rgb_range) for i in idx]
            shapes = {(tuple(p[0].shape), tuple(p[1].shape)) for p in pairs}
            groups = [list(range(len(idx)))] if len(shapes) == 1 else [[j] for j in range(len(idx))]
            for g in groups:                                  # mixed sizes fall back to one image per launch
                order.append([idx[j] for j in g])
                yield (torch.stack([pairs[j][0] for j in g]).pin_memory(), torch.stack([pairs[j][1] for j in g]).pin_memory())

    t_px = t_img = px_above = None
    if cal_files:                                            # calibration pass: maps of the defect-free images, no labels
        cal = metrics.LocalisationAccumulator(n_maps)
        cal_max = []
        with torch.no_grad():
            for _ in ev.run_pipelined(host_batches(cal_files, list(range(len(cal_files))), [])):
                cal.append(ev.last_maps[:-1])                  # device copies, ordered before the next replay overwrites the maps
                cal_max.append(ev.last_maps[-1].clone())
        q = float(calibration_quantile)
        cal_max = torch.cat(cal_max).cpu().numpy()
        t_px = [cal.quantile(j, q) for j in range(n_maps)]
        t_img = [float(np.quantile(cal_max[:, j], q, method='inverted_cdf')) for j in range(n_maps)]
        px_above = [above(t) for t in t_px]
        del cal                                              # the calibration maps are freed before the test pass

    order: List[List[int]] = []
    loc = metrics.LocalisationAccumulator(n_maps) if mask_dir is not None else None   # every map of every image, kept on the device
    test_files = [(e[2], e[3]) for e in entries]
    with torch.no_grad():
        for k, scores in enumerate(ev.run_pipelined(host_batches(test_files, mine, order))):   # PNG decode + H2D of batch k + 1 overlap batch k
            if ev.last_maps is not None:                      # the map maxima ride along in the gathered score table
                scores = torch.cat([scores, ev.last_maps[-1]], 1)
            rows.append(scores)
            ids += order[k]
            if save_images:
                sr_np = ev.last_sr_u8.cpu().numpy()
                for j, i in enumerate(order[k]):
                    name = os.path.splitext(os.path.basename(entries[i][2]))[0]
                    save_sr_image(sr_np[j], output_dir, name, entries[i][1], scale)
            if save_maps:
                host_maps = [m.cpu().numpy() for m in ev.last_maps[:-1]]
                for j, i in enumerate(order[k]):
                    name = os.path.splitext(os.path.basename(entries[i][2]))[0]
                    d = Path(output_dir) / 'maps' / entries[i][1]
                    d.mkdir(parents=True, exist_ok=True)
                    for (kind, _), m in zip(kinds, host_maps):
                        np.save(d / f'{name}_{kind}.npy', m[j])
            if save_calibrated_masks:
                for j, (kind, _) in enumerate(kinds):
                    pred = (ev.last_maps[j] >= px_above[j]).cpu().numpy()
                    for b, i in enumerate(order[k]):
                        name = os.path.splitext(os.path.basename(entries[i][2]))[0]
                        d = Path(output_dir) / 'calibrated' / entries[i][1]
                        d.mkdir(parents=True, exist_ok=True)
                        Image.fromarray(pred[b].astype(np.uint8) * 255).save(str(d / f'{name}_{kind}.png'))
            if loc is not None:
                batch_masks = []
                for i in order[k]:
                    with Image.open(entries[i][3]) as im_lr:
                        crop = (im_lr.size[1] * scale, im_lr.size[0] * scale)
                    batch_masks.append(load_mask(mask_paths[i], tuple(ev.last_maps[0].shape[1:]), crop))
                loc.append(ev.last_maps[:-1], batch_masks)  # device copies, ordered before the next replay overwrites the maps
    n_cols = len(ev.window_sizes) + 2
    local = torch.cat(rows) if rows else torch.empty(0, n_cols + (n_maps if anomaly_maps else 0), dtype=torch.float64, device='cuda')
    table = gather_scores(local, torch.tensor(ids, dtype=torch.int64, device='cuda'), len(entries))
    if table is None:
        return None
    table, map_max = table[:, :n_cols], table[:, n_cols:]
    best_ws, auc_ssim, auc_mse, auc_psnr = metrics.aucs_from_scores(y_true, table, ev.window_sizes)
    res = dict(best_ws=best_ws, auc_ssim=auc_ssim, auc_mse=auc_mse, auc_psnr=auc_psnr, n=len(entries), scores=table)
    if anomaly_maps:
        res['map_max'] = map_max
        for j, (kind, _) in enumerate(kinds):
            res[f'auc_map_{kind}'] = metrics.roc_auc(y_true, map_max[:, j])
        params = {'ssim': f'(ws={map_window_size}, sigma={float(map_sigma)})'}
        line = "Map AUCs - " + ", ".join(f"max {label}{params.get(kind, '')}: {res['auc_map_' + kind]:.4f}" for kind, label in kinds)
        if t_px is not None:
            y = np.asarray(y_true)
            parts = []
            for j, (kind, label) in enumerate(kinds):
                flagged = map_max[:, j] >= above(t_img[j])
                tpr, fpr = float(flagged[y == 1].mean()), float(flagged[y == 0].mean())
                res.update({f'calib_pixel_threshold_{kind}': t_px[j], f'calib_image_threshold_{kind}': t_img[j],
                            f'calib_image_tpr_{kind}': tpr, f'calib_image_fpr_{kind}': fpr})
                part = f"{label} t_px {t_px[j]:g}, t_img {t_img[j]:g}, image TPR {tpr:.4f}, FPR {fpr:.4f}"
                if mask_dir is not None:
                    m = loc.at_threshold(j, px_above[j])
                    res.update({f'calib_pixel_{f}_{kind}': getattr(m, f) for f in ('precision', 'recall', 'fpr', 'f1', 'iou', 'pro')})
                    part += (f", pixel precision {m.precision:.4f}, recall {m.recall:.4f}, FPR {m.fpr:.4f}, F1 {m.f1:.4f}, "
                             f"IoU {m.iou:.4f}, PRO {m.pro:.4f}")
                parts.append(part)
            print(f"Map CAL - q={float(calibration_quantile):g} on {len(cal_files)} defect-free images: " + "; ".join(parts))
        if mask_dir is not None:
            limit = 0.3 if au_pro is None else float(au_pro)
            loc_res = loc.results(limit)                      # one LocalisationMetrics per map kind
            for (kind, _), m in zip(kinds, loc_res):
                res[f'pixel_auroc_{kind}'] = m.pixel_auroc
            line += "".join(f", pixel AUROC {label}: {m.pixel_auroc:.4f}" for (_, label), m in zip(kinds, loc_res))
            if pr_metrics:
                for (kind, _), m in zip(kinds, loc_res):
                    res.update({f'pixel_ap_{kind}': m.pixel_ap, f'f1_max_{kind}': m.f1_max, f'f1_threshold_{kind}': m.f1_threshold})
                print("Map PR - " + ", ".join(f"pixel AP {label}: {m.pixel_ap:.4f}" for (_, label), m in zip(kinds, loc_res)) + ", " +
                      ", ".join(f"F1-max {label}: {m.f1_max:.4f} (thr {m.f1_threshold:g})" for (_, label), m in zip(kinds, loc_res)))
            if save_segmentation:                             # the accumulator holds the images in `ids` order
                for j, ((kind, _), m) in enumerate(zip(kinds, loc_res)):
                    for i, seg in zip(ids, loc.segmentation(j, m.f1_threshold)):
                        name = os.path.splitext(os.path.basename(entries[i][2]))[0]
                        d = Path(output_dir) / 'segmentation' / entries[i][1]
                        d.mkdir(parents=True, exist_ok=True)
                        Image.fromarray(seg.astype(np.uint8) * 255).save(str(d / f'{name}_{kind}.png'))
            if au_pro is not None:
                for (kind, _), m in zip(kinds, loc_res):
                    res[f'au_pro_{kind}'] = m.au_pro
                res['pro_fpr_limit'] = limit
                print("Map PRO - " + ", ".join(f"AU-PRO@{limit:g} {label}: {m.au_pro:.4f}" for (_, label), m in zip(kinds, loc_res)))
        print(line)
    print(f"Test AUCs - SSIM(best ws={best_ws}): {auc_ssim:.4f}, MSE: {auc_mse:.4f}, PSNR: {auc_psnr:.4f}")
    return res


def main(argv=None):
    """src/evaluate.py:270-344."""
    args = parse_args(argv)
    model_type, ds, class_name = args.model_type, args.dataset, args.classe
    img_resolution, scale = args.resolution, args.scale
    if args.run_dir:
        inferred = infer_from_run_dir(args.run_dir)
        model_type = inferred.get('model_type') or model_type
        ds = inferred.get('dataset') or ds
        class_name = inferred.get('classe') or class_name
        img_resolution = inferred.get('resolution') or img_resolution
        scale = inferred.get('scale') or scale
    if args.device in ('cpu', 'mps'):
        raise RuntimeError(f"--device {args.device}: the B200 build has no CPU/MPS path; use the reference for that")
    n_colors = 3 if (ds == 'mvtec' and class_name == 'carpet') else 1
    data_root = args.data_root if args.data_root != 'auto' else f"data/mvtec_{img_resolution}"
    data_dir = f"{data_root}/{class_name}/train/good"
    ckpt_path = resolve_checkpoint(args)
    common = dict(best_auc=0.0, ssim_window_size=11, dataset=ds, classe=class_name, slurm=False, scale=scale,
                  no_augment=True, n_colors=n_colors, epochs=1, batch_size=args.batch_size, patch_size=img_resolution)
    if model_type == 'drn-l':
        opt = setup_opt_drn(DRNOpt(), common['best_auc'], 11, ds, class_name, False, scale, True, n_colors, 1,
                            args.batch_size, img_resolution, data_dir, './workspace/eval', '', 1, 1, 1, 0.0, args.workers,
                            ckpt_path, '.', '1*L1')
    else:
        opt = setup_opt_drct(DRCTOpt(), common['best_auc'], 11, ds, class_name, False, scale, True, n_colors, 1,
                             args.batch_size, img_resolution, img_resolution // scale, data_dir, './workspace/eval', '', 1,
                             1, 1, 0.0, args.workers, ckpt_path, '1*L1')
    opt.model_name, opt.data_root, opt.test_only = model_type, data_root, True
    if 'LOCAL_RANK' in os.environ and int(os.environ.get('WORLD_SIZE', '1')) > 1:
        import torch.distributed as dist

        torch.cuda.set_device(int(os.environ['LOCAL_RANK']))
        dist.init_process_group('nccl')
    out_dir = args.output_dir or (os.path.join(args.run_dir, 'eval_results') if args.run_dir else './workspace/eval_results')
    return evaluate_on_test(opt, ckpt_path, out_dir, args.save_images, batch_size=args.batch_size, anomaly_maps=args.anomaly_maps,
                            map_window_size=args.map_window_size, map_sigma=args.map_sigma, mask_dir=args.mask_dir,
                            save_maps=args.save_maps, au_pro=args.au_pro, pr_metrics=args.pr_metrics,
                            save_segmentation=args.save_segmentation, calibration_dir=args.calibration_dir,
                            calibration_quantile=args.calibration_quantile, save_calibrated_masks=args.save_calibrated_masks,
                            gms_map=args.gms_map)


if __name__ == "__main__":
    main()
