"""Test support: the depth / opacity maps of the compositor and their closed-form backward, built on oracle.port.composite
(whose fp32 / float64 arithmetic the GPU tests already arbitrate with).  The reference computes neither map, so there is no
fixture to pin them against; tests/test_render_maps_cpu.py pins the closed form against float64 autograd of port.composite,
and tests/test_gpu_render.py checks the kernels (hbr_composite_maps_fwd/bwd) against both."""
from __future__ import annotations

from typing import Tuple

import torch

from oracle import port


def composite_maps(t: torch.Tensor, rgb: torch.Tensor, sigma: torch.Tensor, dir_norm):
    """port.composite plus the per-ray maps the project adds (the reference computes neither):
    depth = sum_s w_s t_s (units of t along the unit ray direction; z-depth = depth / dir_norm), opacity = sum_s w_s.
    No normalisation, no clamp.  Returns (C (R,3), w (R,S), depth (R), opacity (R))."""
    C, w = port.composite(t, rgb, sigma, dir_norm)
    tt = t[None, :] if t.dim() == 1 else t
    return C, w, (w * tt).sum(-1), w.sum(-1)


def composite_maps_bwd(t, rgb, sigma, dir_norm, gC, gD, gA) -> Tuple[torch.Tensor, torch.Tensor]:
    """Closed-form backward of composite_maps with per-ray gradients gC (R,3), gD (R), gA (R) of colour, depth and
    opacity: port.composite_bwd with the per-sample term c_k = g.rgb_k + gD t_k + gA (depth and opacity are sums of w_k times
    t_k and 1, exactly as C is the sum of w_k times rgb_k); dL/drgb_k = w_k g is unchanged.
    Returns (d_rgb (R,S,3), d_sigma (R,S))."""
    delta = torch.zeros_like(t)
    delta[..., :-1] = t[..., 1:] - t[..., :-1]
    tt = t[None, :] if t.dim() == 1 else t
    if delta.dim() == 1:
        delta = delta[None, :]
    delta = delta * dir_norm
    keep = sigma >= -10
    p = torch.where(keep, sigma, torch.full_like(sigma, -10.0)) * delta
    e = torch.exp(-p)
    alpha = 1 - e
    Tr = torch.roll(torch.exp(-torch.cumsum(p, dim=-1)), 1, dims=-1)
    Tr = torch.cat([torch.ones_like(Tr[..., :1]), Tr[..., 1:]], dim=-1)
    w = Tr * alpha
    c = (gC[:, None, :] * rgb).sum(-1) + gD[:, None] * tt + gA[:, None]
    wc = w * c
    suffix = torch.flip(torch.cumsum(torch.flip(wc, [-1]), dim=-1), [-1]) - wc
    dp = Tr * e * c - suffix
    return w[..., None] * gC[:, None, :], delta * keep.to(sigma.dtype) * dp
