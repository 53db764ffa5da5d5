"""Test support: float64 restatement of the position gradient of the hash encoding and of the density field, built on
oracle.port (whose hashing and fp32 cell pipeline are pinned bit-exact against the reference).  The reference detaches its
interpolation weights, so it has no position gradient to pin against; tests/test_mesh_cpu.py pins `encode64`'s autograd
against float64 central differences, and tests/test_gpu_mesh.py checks hbr_hash_encode_dx, mesh.field_gradient and
mesh.extract_mesh against this module."""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from oracle import port

_BITS = port._CORNER_BITS                      # (8,3): bit d of corner c


def _level(x_vals, x64, mu, sigma, scale: float, frac_from_fp32: bool):
    """(cell (N,3) int64, frac (N,3) float64, differentiable through the float64 positions x64).  frac_from_fp32: cell and
    frac VALUES from the fp32 pipeline the kernels run at x_vals (port.hash_cells, bit-exact with hbr_hash_indices: no
    cell can disagree), d frac / dx = scale / sigma in float64.  Otherwise a pure float64 evaluation at x64 (for central
    differences)."""
    mu64 = torch.as_tensor(mu, dtype=torch.float64).reshape(-1)
    u = ((x64 - mu64) / float(sigma)) * float(scale)
    if frac_from_fp32:
        cell, fr32 = port.hash_cells(x_vals.detach().float(), torch.as_tensor(mu, dtype=torch.float32).reshape(-1),
                                     torch.tensor(float(sigma), dtype=torch.float32), torch.tensor(float(scale), dtype=torch.float32))
        return cell, fr32.double() + (u - u.detach())
    cell = u.detach().trunc().long()
    return cell, u - cell


def encode64(x64: torch.Tensor, tables: torch.Tensor, mu, sigma, scales, x_vals=None, frac_from_fp32: bool = True):
    """HashEncoder.forward with DIFFERENTIABLE interpolation weights: x64 (N,3) float64 (a leaf with requires_grad for
    autograd), tables (L,T,F) -> (N, L*F) float64, level-major / feature-minor columns.  x_vals: the positions the fp32
    cells / fracs are taken at (default x64 rounded to fp32; pass the caller's fp16 / fp32 tensor)."""
    L, T, F = tables.shape
    t64 = tables.double()
    x_vals = x64.detach().float() if x_vals is None else x_vals
    cols = []
    for l in range(L):
        cell, frac = _level(x_vals, x64, mu, sigma, float(scales[l]), frac_from_fp32)
        idx = port.hash_index(cell[:, None, :] + _BITS[None], T)                       # (N,8)
        fr = frac[:, None, :]
        w = torch.where(_BITS[None].bool(), fr, 1 - fr).prod(dim=-1)                  # (N,8)
        cols.append((t64[l][idx] * w[..., None]).sum(dim=-2))
    return torch.cat(cols, dim=1)


def hash_indices64(x_vals, tables, mu, sigma, scales) -> torch.Tensor:
    """(L,N,8) int64 table indices of the cells encode64 uses (to compare with HashEncoder.hash_indices)."""
    L, T, _ = tables.shape
    out = []
    for l in range(L):
        cell, _ = _level(x_vals, x_vals.double(), mu, sigma, float(scales[l]), True)
        out.append(port.hash_index(cell[:, None, :] + _BITS[None], T))
    return torch.stack(out)


def hash_dx64(x, tables, mu, sigma, scales, dy, frac_from_fp32: bool = True) -> torch.Tensor:
    """dL/dx (N,3) float64 for L = sum(encode64(x) * dy[:, :L*F])."""
    L, _, F = tables.shape
    xx = x.detach().double().clone().requires_grad_(True)
    y = encode64(xx, tables, mu, sigma, scales, x_vals=x, frac_from_fp32=frac_from_fp32)
    (g,) = torch.autograd.grad((y * dy[:, : L * F].double()).sum(), xx)
    return g


def hash_dx_magnitude(x, tables, mu, sigma, scales, dy) -> torch.Tensor:
    """(N,3) float64: sum over levels, corners and features of |s_l/sigma| |dy_f v_cf| prod_{b != a} |w_b| -- the size of
    the terms dx_a is a sum of (the yardstick of an element-wise bound; dx itself may cancel)."""
    L, T, F = tables.shape
    t64 = tables.double()
    out = torch.zeros(x.shape[0], 3, dtype=torch.float64)
    for l in range(L):
        s = float(scales[l])
        cell, frac = _level(x, x.double(), mu, sigma, s, True)
        frac = frac.detach()
        idx = port.hash_index(cell[:, None, :] + _BITS[None], T)
        gabs = (t64[l][idx].abs() * dy[:, None, l * F:(l + 1) * F].double().abs()).sum(-1)      # (N,8)
        fr = frac[:, None, :]
        w = torch.where(_BITS[None].bool(), fr, 1 - fr).abs()                              # (N,8,3)
        for a in range(3):
            others = [b for b in range(3) if b != a]
            out[:, a] += abs(s / float(sigma)) * (gabs * w[..., others[0]] * w[..., others[1]]).sum(-1)
    return out


def _p64(p_mlp: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    return {k: v.detach().double().cpu() for k, v in p_mlp.items()}


def field_gradient64(p_mlp, tables, mu, sigma, scales, x) -> Tuple[torch.Tensor, torch.Tensor]:
    """(density (N,), grad (N,3)) float64: port.mlp_forward's density column through encode64, differentiated by autograd
    (the LeakyReLU slope included).  Cells and fracs are the fp32 pipeline's values at x."""
    xx = x.detach().double().clone().requires_grad_(True)
    feat = encode64(xx, tables, mu, sigma, scales, x_vals=x)
    dens = port.mlp_forward(_p64(p_mlp), feat, None)[:, 0]
    (g,) = torch.autograd.grad(dens.sum(), xx)
    return dens.detach(), g


def colors64(p_mlp, tables, mu, sigma, scales, x, view_dirs, num_freq: int = 4) -> torch.Tensor:
    """(N,3) float64 raw RGB of the full field at x seen along view_dirs (N,3) (encoded with port.dir_encode)."""
    feat = encode64(x.detach().double(), tables, mu, sigma, scales, x_vals=x)
    return port.mlp_forward(_p64(p_mlp), feat, port.dir_encode(view_dirs.double(), num_freq))[:, :3]


def relu_margin64(p_mlp, tables, mu, sigma, scales, x) -> torch.Tensor:
    """(N,) float64: min over the density head's hidden ReLU units of |pre-activation| / (sum_k |W_jk a_k| + |b_j|).  The
    field's gradient jumps where a pre-activation crosses zero, so where this is at rounding level an fp32 evaluation may
    legitimately sit on the other side of the kink."""
    p = _p64(p_mlp)
    h = encode64(x.detach().double(), tables, mu, sigma, scales, x_vals=x).detach()
    m = torch.full((x.shape[0],), float("inf"), dtype=torch.float64)
    for i in (0, 2):
        W, b = p[f"sig_model.{i}.weight"], p[f"sig_model.{i}.bias"]
        z = h @ W.T + b
        m = torch.minimum(m, (z.abs() / (h.abs() @ W.abs().T + b.abs())).min(dim=1).values)
        h = torch.relu(z)
    return m
