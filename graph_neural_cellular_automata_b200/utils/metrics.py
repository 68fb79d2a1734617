"""The trainer's per-step quality metrics on the device (train_graph_augmented_nca.py:405-422 computes them with
numpy/skimage on sample 0 after a host copy): pixel-perfection, PSNR and SSIM on premultiplied RGBA, for the whole
batch, without leaving the GPU.  SSIM is one library call (gnca_ssim_rgb); the others are torch expressions."""
from __future__ import annotations

import ctypes as C

import torch


def premultiply(state: torch.Tensor) -> torch.Tensor:
    pred = state[:, :4]
    return torch.cat([pred[:, :3] * pred[:, 3:4], pred[:, 3:4]], dim=1)


def pixel_perfect(state: torch.Tensor, target: torch.Tensor, eps: float = 0.05) -> torch.Tensor:
    """fraction of pixels whose 4 premultiplied RGBA channels are all within eps of the target; per sample [B]"""
    diff = (premultiply(state) - target.unsqueeze(0)).abs()
    return (diff < eps).all(dim=1).float().mean(dim=(1, 2))


def psnr_rgb(state: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """skimage.metrics.peak_signal_noise_ratio(data_range=1) on the clipped premultiplied RGB; per sample [B]"""
    a = premultiply(state)[:, :3].clamp(0, 1)
    b = target[:3].unsqueeze(0).clamp(0, 1)
    mse = ((a - b) ** 2).mean(dim=(1, 2, 3))
    return 10.0 * torch.log10(1.0 / mse)


def ssim_rgb(state: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """skimage.metrics.structural_similarity(pred, tgt, channel_axis=-1, data_range=1.0), every other argument at its
    default, per sample [B] float32, on the device (gnca_ssim_rgb; no CPU fallback).

    pred = clip(premultiplied RGB of the state, 0, 1), tgt = clip(target RGB, 0, 1): the images of psnr_rgb.  Per
    channel: 7x7 uniform windows, window means ux, uy, covariances vx, vy, vxy with cov_norm = 49/48, C1 = 0.01^2,
    C2 = 0.03^2, S = (2 ux uy + C1)(2 vxy + C2) / ((ux^2 + uy^2 + C1)(vx + vy + C2)), averaged over the (H-6)(W-6)
    interior cells (skimage crops a 3-cell border, so every window lies inside the grid); the SSIM is the mean of the
    three channel means.  The window moments are taken in double, summed in a fixed order: two calls give the same bits.

    state: [B, C >= 4, H, W] fp32 (alpha = channel 3); target: [4, H, W] premultiplied RGBA on the same device.
    H or W below 7 raises ValueError, as skimage does."""
    from .. import _lib
    from .. import functional as GF
    if state.dim() != 4 or state.shape[1] < 4:
        raise ValueError(f"ssim_rgb: state must be [B, C >= 4, H, W], got {list(state.shape)}")
    B, Cc, H, W = state.shape
    if tuple(target.shape) != (4, H, W):
        raise ValueError(f"ssim_rgb: target must be [4, {H}, {W}] (premultiplied RGBA), got {list(target.shape)}")
    if H < 7 or W < 7:
        raise ValueError(f"ssim_rgb: SSIM needs a 7x7 window inside the grid, got H={H}, W={W}")
    if B == 0:
        raise ValueError("ssim_rgb: empty batch")
    x = GF._require_cuda_f32(state.detach(), "state")
    tgt = GF._require_cuda_f32(target.detach(), "target")
    if tgt.device != x.device:
        raise ValueError(f"ssim_rgb: target is on {tgt.device}, state on {x.device}")
    lib = _lib.load()
    out = torch.empty(B, dtype=torch.float64, device=x.device)
    scratch = torch.empty(lib.gnca_ssim_rgb_scratch_bytes(B, H, W), dtype=torch.uint8, device=x.device)
    _lib.check(lib.gnca_ssim_rgb(GF._ptr(x), B, Cc, H, W, GF._ptr(tgt), GF._ptr(out), GF._ptr(scratch),
                                 C.c_size_t(scratch.numel()), GF._stream()), "gnca_ssim_rgb")
    return out.float()
