"""fp64 restatement of the SSIM the library computes (utils.metrics.ssim_rgb, monitor_rollout(..., ssim=True)).

SSIM is skimage.metrics.structural_similarity(pred, tgt, channel_axis=-1, data_range=1.0) with every other argument
at its default, on pred = clip(premultiplied RGB of the state, 0, 1) and tgt = clip(target RGB, 0, 1).  The state is
premultiplied in fp32 (r * alpha, alpha = channel 3), as utils.metrics does, and everything after that is float64:

- per channel, 7x7 uniform windows: window means ux, uy; vx = cov_norm (E[x^2] - ux^2), vy likewise,
  vxy = cov_norm (E[xy] - ux uy), cov_norm = 49/48;
- C1 = 0.01^2, C2 = 0.03^2, S = (2 ux uy + C1)(2 vxy + C2) / ((ux^2 + uy^2 + C1)(vx + vy + C2));
- the mean of S over the (H-6)(W-6) interior cells (skimage crops a border of 3, so every window lies inside the grid
  and no padding mode enters); SSIM = the mean of the three channel means.
H or W below 7 raises ValueError, as skimage does."""
from __future__ import annotations

import numpy as np
import torch

WIN = 7
C1, C2 = 0.01 ** 2, 0.03 ** 2


def images(state: torch.Tensor, target: torch.Tensor):
    """(pred [B,3,H,W], tgt [3,H,W]) in float64: the clipped premultiplied RGB, rounded in fp32 first"""
    s = state.detach().cpu().float()
    pred = (s[:, :3] * s[:, 3:4]).clamp(0, 1).double().numpy()
    tgt = target.detach().cpu().float()[:3].clamp(0, 1).double().numpy()
    return pred, tgt


def ssim_rgb(state: torch.Tensor, target: torch.Tensor) -> np.ndarray:
    """[B] float64 SSIM of the states [B, C >= 4, H, W] against the premultiplied target [4, H, W]"""
    H, W = state.shape[-2:]
    if H < WIN or W < WIN:
        raise ValueError(f"SSIM needs a {WIN}x{WIN} window inside the grid, got {H}x{W}")
    pred, tgt = images(state, target)
    win = lambda a: np.lib.stride_tricks.sliding_window_view(a, (WIN, WIN), axis=(-2, -1)).mean(axis=(-2, -1))
    x, y = pred, tgt[None]
    ux, uy = win(x), win(y)
    cov_norm = WIN * WIN / (WIN * WIN - 1.0)
    vx = cov_norm * (win(x * x) - ux * ux)
    vy = cov_norm * (win(y * y) - uy * uy)
    vxy = cov_norm * (win(x * y) - ux * uy)
    S = (2 * ux * uy + C1) * (2 * vxy + C2) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))
    return S.mean(axis=(-2, -1)).mean(axis=-1)          # interior cells per channel, then the three channels
