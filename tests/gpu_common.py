"""Helpers shared by the `-m gpu` parity tests (no reads of /root/reference at run time)."""
import importlib

import torch

PKG = "anomaly-detection-super-resolution_b200"

# the torch side of every comparison must be true fp32 (no TF32 in cuDNN / cuBLAS)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def mod(name):
    return importlib.import_module(f"{PKG}.{name}")


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).float()


def rel_err(got: torch.Tensor, want: torch.Tensor) -> float:
    return float((got.float() - want.float()).abs().max() / want.float().abs().max().clamp_min(1e-12))


class DrctOpt:
    """Same fields the reference's DRCT dataclass carries (src/main.py:83-142), filled like setup_opt_drct."""

    def __init__(self, img_size=32, n_colors=3, embed_dim=180, layers=12, heads=6, upscale=4, rgb_range=255):
        self.img_size, self.n_colors, self.embed_dim = img_size, n_colors, embed_dim
        self.depths = (6,) * layers
        self.num_heads = (heads,) * layers
        self.window_size = img_size // 4
        self.mlp_ratio, self.upscale, self.img_range = 2, upscale, 1.0
        self.upsampler, self.resi_connection, self.rgb_range = "pixelshuffle", "1conv", rgb_range
        self.compress_ratio, self.squeeze_factor, self.conv_scale, self.overlap_ratio = 3, 30, 0.01, 0.5
        self.scale = [upscale]


class TableModel:
    """Stands in for the SR network: `run` returns precomputed uint8 SR images for the LR batch it is handed (the LR tensor's
    first element carries the index of the batch's first image), so the evaluator's batching, scoring, gather and AUC logic can
    be driven over a large image set without a forward pass."""

    def __init__(self, sr_u8: torch.Tensor):
        self.sr_u8 = sr_u8

    def run(self, lr_d, want_float=False, want_u8=True):
        i0 = int(lr_d[0, 0, 0, 0].item())
        return None, self.sr_u8[i0:i0 + lr_d.shape[0]]
