"""TEST INFRASTRUCTURE ONLY: CPU restatement ("port") of the reference NeRF hot path.

Nothing in the product package may import this module.  It exists so that the CUDA path
can be checked without a checkout of the reference.  Allowed
importers: tests/, __graft_entry__.smoke(), and bench.py's cpu_baseline / --impl reference legs.

Parity status: PINNED.  The reference ships no tests or golden vectors (SURVEY.md section 4),
so every function here is pinned against outputs of the reference itself, executed in the
build container by oracle/make_golden.py (fixtures committed in tests/golden/*.npz) and, when
the reference tree is present, live in tests/test_oracle_golden.py.
Exception: marching cubes (torchmcubes==0.1.0, Nerf.yml:198, source not vendored) -- only the
table-independent invariant "welded vertex count == number of iso-crossing grid edges" is
pinned; vertex order / face lists are parity-unpinned (see DESIGN.md).

All arithmetic is torch-on-CPU fp32 in the reference's operation order (true division, no FMA
contraction, truncating .long()), so the integer results (cells, hash indices) are bit-exact
and the floating point results are reproducible.  Pass dtype=torch.float64 where offered to
arbitrate fp32 ordering disputes.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as Fnn

# hash_encoding.py:24 -- np.array([1, 2654435761, 805459861], dtype=np.int32) under numpy 1.x
PRIMES = (1, -1640531535, 805459861)


# ------------------------------------------------------------------------------------------------
# a1/a2/a3/a4: multiresolution hash encoder
# ------------------------------------------------------------------------------------------------
def level_scales(n_min, n_max, L: int) -> torch.Tensor:
    """Per-level grid scales N_l = N_min * b**l, b = exp((ln N_max - ln N_min)/(L-1)).

    hash_encoding.py:11-13 (b) and :153 (N_l).  Non-integer fp32, evaluated with torch CPU scalars
    exactly as the reference does on every forward call (SURVEY Q1/Q2)."""
    N_max = torch.tensor(n_max)
    N_min = torch.tensor(n_min)
    b = torch.exp((torch.log(N_max) - torch.log(N_min)) / (L - 1))
    return torch.stack([(N_min * b ** i).to(torch.float32).reshape(()) for i in range(L)])


def hash_index(corner: torch.Tensor, T: int) -> torch.Tensor:
    """Spatial hash of integer lattice corners (..., 3) int64 -> (...) int64 in [0, T).

    hash_encoding.py:49-53: int64 products with the int32 primes, XOR, Python-style (floor) modulo."""
    pis = torch.tensor(PRIMES, dtype=torch.int64)
    prod = corner.to(torch.int64) * pis
    v = torch.bitwise_xor(torch.bitwise_xor(prod[..., 0], prod[..., 1]), prod[..., 2])
    return torch.remainder(v, T)


def hash_index_u32_pow2(corner: np.ndarray, T: int) -> np.ndarray:
    """The uint32 form the CUDA kernel uses for power-of-two T (SURVEY Q5); numpy, for cross-checks."""
    assert T & (T - 1) == 0
    c = corner.astype(np.int64).astype(np.uint32)  # low 32 bits, two's complement
    with np.errstate(over="ignore"):
        h = c[..., 0] ^ (c[..., 1] * np.uint32(2654435761)) ^ (c[..., 2] * np.uint32(805459861))
    return (h & np.uint32(T - 1)).astype(np.int64)


_CORNER_BITS = torch.tensor([[(c >> d) & 1 for d in range(3)] for c in range(8)], dtype=torch.int64)  # (8,3)


def hash_cells(x: torch.Tensor, mu, sigma, scale) -> Tuple[torch.Tensor, torch.Tensor]:
    """Cell index and in-cell fraction at one level.  hash_encoding.py:154-158.

    un_x = ((x - mu) / sigma) * N_l, each op rounded separately in fp32 (fp16 x is promoted by the
    subtraction); x0 = trunc toward zero (.long()); frac = un_x - x0 (may be negative for un_x < 0)."""
    un_x = ((x - mu) / sigma) * scale
    x0 = un_x.long()
    frac = un_x - x0
    return x0, frac


def hash_level_aux(x, mu, sigma, scale, T):
    """(idx (N,8) int64, w (N,8) float) for one level: corner c takes x0+1 in dim d iff bit d of c
    (hash_encoding.py:34-37,135); weight = prod_d (bit ? frac : 1-frac) in x,y,z order (:142-143)."""
    x0, frac = hash_cells(x, mu, sigma, scale)
    corners = x0[:, None, :] + _CORNER_BITS[None]                      # (N,8,3)
    idx = hash_index(corners, T)
    fr = frac[:, None, :]
    sel = _CORNER_BITS[None].bool()
    w = torch.where(sel, fr, 1 - fr).prod(dim=-1)                       # (N,8)
    return idx, w


def hash_encode(x: torch.Tensor, tables: torch.Tensor, mu, sigma, scales: torch.Tensor, E: int = 0,
                return_aux: bool = False):
    """HashEncoder.forward (hash_encoding.py:146-170).

    x (N,3) fp32|fp16, tables (L,T,F) fp32 -> y (N, L*F+E) fp32, level-major / feature-minor columns,
    E trailing zero columns.  With return_aux also returns idx (L,N,8) int64 and w (L,N,8)."""
    L, T, F = tables.shape
    N = x.shape[0]
    y = torch.zeros(N, L * F + E, dtype=tables.dtype)
    idxs, ws = [], []
    for l in range(L):
        idx, w = hash_level_aux(x, mu, sigma, scales[l], T)
        fv = tables[l][idx]                                             # (N,8,F)   :163
        y[:, l * F:(l + 1) * F] = (fv * w[..., None].to(fv.dtype)).sum(dim=-2)   # :144,165
        if return_aux:
            idxs.append(idx)
            ws.append(w)
    if return_aux:
        return y, torch.stack(idxs), torch.stack(ws)
    return y


def hash_encode_bwd(dy: torch.Tensor, idx: torch.Tensor, w: torch.Tensor, T: int, F: int,
                    dtype=torch.float64) -> torch.Tensor:
    """Table gradient dtable[l, h] += w * dy[:, lF:(l+1)F] over all 8 corners (autograd of
    hash_encoding.py:163-165; nn.Embedding(sparse=False) -> dense grads; no grad to x because
    diff is detached at :160).  Accumulates in `dtype` (fp64 by default: the arbitration value)."""
    L = idx.shape[0]
    g = torch.zeros(L, T, F, dtype=dtype)
    for l in range(L):
        contrib = w[l][..., None].to(dtype) * dy[:, None, l * F:(l + 1) * F].to(dtype)   # (N,8,F)
        g[l].index_add_(0, idx[l].reshape(-1), contrib.reshape(-1, F))
    return g


# ------------------------------------------------------------------------------------------------
# a6: direction encoding
# ------------------------------------------------------------------------------------------------
def dir_encode(d: torch.Tensor, num_freq: int) -> torch.Tensor:
    """PositionalEncoder.forward (encoder.py:25-32): per component [sin(2 x k)]_k || [cos(2 x k)]_k,
    k = 0..num_freq-1 (linear k, int8 tensor), flattened to (N, dim*2*num_freq) as the callers do
    (vol_renderer.py:183)."""
    k = torch.arange(0, num_freq, dtype=torch.int8)[None, None, :]
    a = 2 * d.unsqueeze(-1) * k
    out = torch.cat([torch.sin(a), torch.cos(a)], dim=-1)
    return out.reshape(out.shape[0], -1)


# ------------------------------------------------------------------------------------------------
# a7: MLP_3D
# ------------------------------------------------------------------------------------------------
MLP_KEYS = ("sig_model.0", "sig_model.2", "sig_model.4", "col_model.0", "col_model.2", "col_model.4")


def mlp_shapes(L=16, F=2, E=0, d_view=24, h=64):
    """(out,in) of the six Linear layers for MLP_3D(num_sig=2,num_col=2) (test_hash.py:27-50)."""
    return {"sig_model.0": (h, L * F + E), "sig_model.2": (h, h), "sig_model.4": (16, h),
            "col_model.0": (h, 15 + d_view), "col_model.2": (h, h), "col_model.4": (3, h)}


def mlp_init(seed: int = 0, **kw) -> Dict[str, torch.Tensor]:
    """nn.Linear default init, in module construction order (so it equals MLP_3D under the same seed)."""
    g = torch.Generator().manual_seed(seed)
    p = {}
    for k, (o, i) in mlp_shapes(**kw).items():
        bound = 1.0 / math.sqrt(i)
        p[k + ".weight"] = (torch.rand(o, i, generator=g) * 2 - 1) * bound
        p[k + ".bias"] = (torch.rand(o, generator=g) * 2 - 1) * bound
    return p


def mlp_forward(p: Dict[str, torch.Tensor], feat: torch.Tensor, dirs: Optional[torch.Tensor]) -> torch.Tensor:
    """MLP_3D.forward, NeRF mode (test_hash.py:52-77).

    sigma-net Linear-ReLU-Linear-ReLU-Linear(16); density = LeakyReLU_0.01(out[:,0:1]); colour-net on
    cat(out[:,1:], dirs): Linear-ReLU-Linear-ReLU-Linear(3); rgb = ELU(.); returns cat(rgb, density) (N,4).
    With dirs=None returns the density column only (N,1)."""
    h = Fnn.relu(Fnn.linear(feat, p["sig_model.0.weight"], p["sig_model.0.bias"]))
    h = Fnn.relu(Fnn.linear(h, p["sig_model.2.weight"], p["sig_model.2.bias"]))
    dens_vec = Fnn.linear(h, p["sig_model.4.weight"], p["sig_model.4.bias"])
    density = Fnn.leaky_relu(dens_vec[:, 0:1], 0.01)
    if dirs is None:
        return density
    c = torch.cat((dens_vec[:, 1:], dirs.to(dens_vec.dtype)), dim=-1)
    c = Fnn.relu(Fnn.linear(c, p["col_model.0.weight"], p["col_model.0.bias"]))
    c = Fnn.relu(Fnn.linear(c, p["col_model.2.weight"], p["col_model.2.bias"]))
    rgb = Fnn.elu(Fnn.linear(c, p["col_model.4.weight"], p["col_model.4.bias"]))
    return torch.cat((rgb, density), dim=-1)


# ------------------------------------------------------------------------------------------------
# a8-a11: sampling and compositing
# ------------------------------------------------------------------------------------------------
def strat_t(near, far, S: int, u: torch.Tensor) -> torch.Tensor:
    """strat_sampler, linear branch (helper.py:234-235): t = linspace(tn,tf,S) + u*(tf-tn)/S with
    u = rand_like(t) passed in (RNG draw #1 of a vol_render call, SURVEY Q9)."""
    t = torch.linspace(near, far, S)
    return t + (u * (far - near) / S)


def ray_points(rays_o, rays_d, t):
    """vol_renderer.py:165 / helper.py:48: o + d*t with a separate multiply and add.
    t is (S,) shared by all rays or (R,S) per ray."""
    tt = t[None, :, None] if t.dim() == 1 else t[..., :, None]
    return rays_o[..., None, :] + rays_d[..., None, :] * tt


def composite(t: torch.Tensor, rgb: torch.Tensor, sigma: torch.Tensor, dir_norm) -> Tuple[torch.Tensor, torch.Tensor]:
    """calc_color, NeRF mode (helper.py:65-107).  Does NOT modify its inputs (the reference clamps
    sigma in place at :76; callers that depend on that side effect must clamp themselves).

    delta[:-1] = t[1:]-t[:-1], delta[-1] = 0, times dir_norm (R,1); sigma clamped below at -10;
    p = sigma*delta; alpha = 1-exp(-p); T = exclusive exp(-cumsum(p)); w = T*alpha; C = sum_s w*rgb.
    Returns (C (R,3), w (R,S))."""
    delta = torch.zeros_like(t)
    delta[..., :-1] = t[..., 1:] - t[..., :-1]
    if delta.dim() == 1:
        delta = delta[None, :]
    delta = delta * dir_norm
    sig = torch.where(sigma < -10, torch.full_like(sigma, -10.0), sigma)
    p = sig * delta
    alpha = 1 - torch.exp(-p)
    Tr = torch.exp(-torch.cumsum(p, dim=-1))
    Tr = torch.roll(Tr, 1, dims=-1)
    Tr = torch.cat([torch.ones_like(Tr[..., :1]), Tr[..., 1:]], dim=-1)
    w = Tr * alpha
    C = torch.sum(w[..., None] * rgb, dim=-2)
    return C, w


def composite_bwd(t, rgb, sigma, dir_norm, gC) -> Tuple[torch.Tensor, torch.Tensor]:
    """Closed-form backward of `composite` (SURVEY appendix A.3), same dtype as the inputs.

    dL/drgb_k = w_k g;  c_k = g.rgb_k;  dL/dp_k = T_k (1-alpha_k) c_k - sum_{i>k} w_i c_i;
    dL/dsigma_k = delta_k [sigma_k >= -10] dL/dp_k.   Returns (d_rgb (R,S,3), d_sigma (R,S))."""
    delta = torch.zeros_like(t)
    delta[..., :-1] = t[..., 1:] - t[..., :-1]
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
    c = (gC[:, None, :] * rgb).sum(-1)
    wc = w * c
    suffix = torch.flip(torch.cumsum(torch.flip(wc, [-1]), dim=-1), [-1]) - wc
    dp = Tr * e * c - suffix
    return w[..., None] * gC[:, None, :], delta * keep.to(sigma.dtype) * dp


def hier_sample(wts: torch.Tensor, t: torch.Tensor, near, far, u_rs: torch.Tensor, u_s: torch.Tensor) -> torch.Tensor:
    """hierarchical_sampling (helper.py:36-47) with the two uniform draws passed in
    (u_rs = rand(R,S) draw #2, u_s = rand(S) draw #3, SURVEY Q9).  Returns combined depths (R,2S), sorted.

    w<0 -> 0; pdf=(w+1e-5)/sum; cdf=cumsum; inds=searchsorted(cdf,u,right=True) clamped to S-1;
    ONE shared unsorted vector of S candidate depths u_s*(tf-tn)+tn, gathered by inds; merged with the
    S coarse depths and sorted."""
    w = torch.where(wts < 0, torch.zeros_like(wts), wts)
    pdf = (w + 1e-5) / torch.sum(w + 1e-5, dim=-1, keepdim=True)
    cdf = torch.cumsum(pdf, dim=-1)
    inds = torch.searchsorted(cdf, u_rs, right=True)
    cand = u_s * (far - near) + near
    inds = torch.clamp(inds, min=0, max=cand.shape[-1] - 1)
    fine = cand[inds]
    z = t.expand(list(inds.shape[:-1]) + [t.shape[-1]])
    merged, _ = torch.sort(torch.cat([z, fine], dim=-1), dim=-1)
    return merged


def occupancy_mask(points: torch.Tensor, bool_grid: torch.Tensor, mu, sigma_val) -> torch.Tensor:
    """Volume_Renderer.get_mask (vol_renderer.py:133-140): bool_grid[((p-mu)/sigma*G).long()]
    (negative cells wrap like Python indexing)."""
    G = bool_grid.shape[0]
    q = ((points - mu) / sigma_val) * G
    q = q.long()
    return bool_grid[q[..., 0], q[..., 1], q[..., 2]]


def vol_render(p_mlp, tables, mu, sigma, scales, rays_d, rays_o, t, dir_norm, num_freq=4,
               hierarchical=False, near=None, far=None, u_rs=None, u_s=None, bool_grid=None,
               update_mask=False, t_fine=None):
    """Volume_Renderer.vol_render (vol_renderer.py:141-245), NeRF mode, with the strat depths `t`
    and the hierarchical draws supplied.  Returns (Cr, Cf, aux) with aux = dict(w=..., t_fine=...).
    t_fine: use these fine depths instead of resampling (the depths carry no gradient, helper.py:41-47: searchsorted /
    gather / sort of detached values) -- lets a test evaluate the reference's fine pass and its gradients on the sampling
    decisions of the implementation under test, whose coarse weights differ from the CPU's in the last bits."""
    R, S = rays_o.shape[0], t.shape[0]
    pts = ray_points(rays_o, rays_d, t).reshape(-1, 3)
    dirs = dir_encode(rays_d[:, None, :].repeat(1, S, 1).reshape(-1, 3), num_freq)
    feat = hash_encode(pts, tables, mu, sigma, scales)
    out = mlp_forward(p_mlp, feat, dirs)
    if (not update_mask) and bool_grid is not None:
        m = occupancy_mask(pts, bool_grid, mu, sigma)       # vol_renderer.py:211-216: masked-out samples are 0
        out = out * m[:, None].to(out.dtype)
    sig = out[:, 3].reshape(R, S)
    rgb = out[:, 0:3].reshape(R, S, 3)
    Cr, w = composite(t, rgb, sig, dir_norm)
    aux = {"w": w}
    if not hierarchical:
        return Cr, Cr, aux
    if t_fine is None:
        t_fine = hier_sample(w.detach(), t, near, far, u_rs, u_s)
    pts_f = ray_points(rays_o, rays_d, t_fine).reshape(-1, 3)
    dirs_f = dir_encode(rays_d[:, None, :].repeat(1, 2 * S, 1).reshape(-1, 3), num_freq)
    out_f = mlp_forward(p_mlp, hash_encode(pts_f, tables, mu, sigma, scales), dirs_f)
    Cf, _ = composite(t_fine, out_f[:, 0:3].reshape(R, 2 * S, 3), out_f[:, 3].reshape(R, 2 * S), dir_norm)
    aux["t_fine"] = t_fine
    return Cr, Cf, aux


# ------------------------------------------------------------------------------------------------
# SDF mode (8f row 4): test_hash.py:59-60,78-105; helper.py:13-21,76-89,102-107,293-299
# ------------------------------------------------------------------------------------------------
def mlp_forward_sdf(p: Dict[str, torch.Tensor], feat: torch.Tensor, dirs: Optional[torch.Tensor]) -> torch.Tensor:
    """MLP_3D.forward with use_sdf=True (test_hash.py:59-60): the density column is 2*sigmoid(dens_vec[:,0:1]) - 1
    instead of LeakyReLU; dirs=None gives forward_sdf's value (test_hash.py:78-84)."""
    h = Fnn.relu(Fnn.linear(feat, p["sig_model.0.weight"], p["sig_model.0.bias"]))
    h = Fnn.relu(Fnn.linear(h, p["sig_model.2.weight"], p["sig_model.2.bias"]))
    dens_vec = Fnn.linear(h, p["sig_model.4.weight"], p["sig_model.4.bias"])
    sdf = 2 * torch.sigmoid(dens_vec[:, 0:1]) - 1
    if dirs is None:
        return sdf
    c = torch.cat((dens_vec[:, 1:], dirs.to(dens_vec.dtype)), dim=-1)
    c = Fnn.relu(Fnn.linear(c, p["col_model.0.weight"], p["col_model.0.bias"]))
    c = Fnn.relu(Fnn.linear(c, p["col_model.2.weight"], p["col_model.2.bias"]))
    rgb = Fnn.elu(Fnn.linear(c, p["col_model.4.weight"], p["col_model.4.bias"]))
    return torch.cat((rgb, sdf), dim=-1)


def fd_normals(p_mlp, tables, mu, sigma, scales, x, min_bound, max_bound, epsilon: float = 0.0005) -> torch.Tensor:
    """MLP_3D.finite_difference_normals_approximator (test_hash.py:86-105): central differences of forward_sdf at
    positions clamped to the bounding box."""
    cols = []
    for axis in range(3):
        e = torch.zeros(1, 3)
        e[0, axis] = epsilon
        pos = mlp_forward_sdf(p_mlp, hash_encode((x + e).clamp(min_bound, max_bound), tables, mu, sigma, scales), None)
        neg = mlp_forward_sdf(p_mlp, hash_encode((x - e).clamp(min_bound, max_bound), tables, mu, sigma, scales), None)
        cols.append(0.5 * (pos - neg) / epsilon)
    return torch.cat(cols, dim=-1)


def composite_sdf(rgb: torch.Tensor, sdf: torch.Tensor, b) -> Tuple[torch.Tensor, torch.Tensor]:
    """calc_color, SDF branch (helper.py:76-86,102-105) on a COPY of sdf (R,S): clamp at -10, phi = 1/(1+exp(-s*b))
    (VarModel, helper.py:18-21), alpha_i = relu(1 - phi_{i+1}/phi_i) (last sample 0), T = exclusive cumprod(1-alpha).
    Returns (Cr (R,3), wts (R,S,1))."""
    s = sdf.clone()
    s[s < -10] = -10
    phi = 1 / (1 + torch.exp(-s * b))
    alpha = torch.zeros_like(s)
    alpha[..., :-1] = 1 - phi[..., 1:] / phi[..., :-1]
    alpha = Fnn.relu(alpha)
    T = torch.roll(torch.cumprod(1 - alpha, -1), 1, -1)
    T[..., 0] = 1.0
    wts = T[:, :, None] * alpha[:, :, None]
    return torch.sum(T[:, :, None] * alpha[:, :, None] * rgb, dim=-2), wts


def composite_sdf_bwd(rgb: torch.Tensor, sdf: torch.Tensor, b, gC: torch.Tensor, gw: Optional[torch.Tensor] = None):
    """Closed-form backward of composite_sdf (what autograd gives for helper.py:76-86,102-105), the derivation the CUDA
    kernel follows: with c_i = gC . rgb_i + gw_i, r_i = phi_{i+1} / phi_i, suffix_i = sum_{k>i} w_k c_k,
      e_i = alpha_i > 0 ? suffix_i - T_i c_i (1 - alpha_i) : 0        (= dL/dr_i * r_i; relu'(0) = 0)
      dL/d(s_i b) = (1 - phi_i) (e_{i-1} - e_i),   e_{-1} = e_{S-1} = 0
    Returns (d rgb (R,S,3), d sdf (R,S) -- 0 where the -10 clamp hit --, dL/db scalar)."""
    s = sdf.clone()
    keep = ~(s < -10)
    s[~keep] = -10
    phi = 1 / (1 + torch.exp(-s * b))
    r = torch.ones_like(s)
    r[..., :-1] = phi[..., 1:] / phi[..., :-1]
    alpha = torch.clamp(1 - r, min=0)
    alpha[..., -1] = 0
    T = torch.ones_like(s)
    T[..., 1:] = torch.cumprod(1 - alpha, -1)[..., :-1]
    w = T * alpha
    c = (rgb * gC[:, None, :]).sum(-1)
    if gw is not None:
        c = c + gw
    wc = w * c
    suffix = torch.flip(torch.cumsum(torch.flip(wc, [-1]), -1), [-1]) - wc
    e = torch.where(alpha > 0, suffix - T * c * (1 - alpha), torch.zeros_like(s))
    e_prev = torch.zeros_like(e)
    e_prev[..., 1:] = e[..., :-1]
    base = (1 - phi) * (e_prev - e)
    return w[..., None] * gC[:, None, :], torch.where(keep, b * base, torch.zeros_like(s)), (s * base).sum()


def vol_render_sdf(p_mlp, tables, mu, sigma, scales, rays_d, rays_o, t, b, min_bound, max_bound, num_freq=4):
    """Volume_Renderer.vol_render with use_sdf=True, hierarchical=False, all-True occupancy grid
    (vol_renderer.py:165-223 -> helper.py:80-89).  Returns (Cr, wts, eikonal norms (R*S,))."""
    R, S = rays_o.shape[0], t.shape[0]
    pts = ray_points(rays_o, rays_d, t).reshape(-1, 3)
    dirs = dir_encode(rays_d[:, None, :].repeat(1, S, 1).reshape(-1, 3), num_freq)
    out = mlp_forward_sdf(p_mlp, hash_encode(pts, tables, mu, sigma, scales), dirs)
    Cr, wts = composite_sdf(out[:, 0:3].reshape(R, S, 3), out[:, 3].reshape(R, S), b)
    grads = fd_normals(p_mlp, tables, mu, sigma, scales, pts, min_bound, max_bound)
    return Cr, wts, torch.sqrt(torch.sum(grads ** 2, dim=-1))


# ------------------------------------------------------------------------------------------------
# callers' setup either side of the path (rows "next": get_od, find_bounding_box)
# ------------------------------------------------------------------------------------------------
def get_od(H: int, W: int, K: torch.Tensor, c2w: torch.Tensor):
    """helper.py:176-208.  K is the int64 intrinsics matrix of train_hash2.py:67-72 (focal truncated, Q14).
    c2w (B,4,4).  Returns rays_o (B,HW,3), unit rays_d (B,HW,3), dir_norm (B,HW,1)."""
    i, j = torch.meshgrid(torch.arange(W), torch.arange(H), indexing="xy")
    i = ((i - K[0, 2]) / K[0, 0]).reshape(-1)
    j = ((j - K[1, 2]) / K[1, 1]).reshape(-1)
    dirs = torch.stack((i, -j, -torch.ones_like(i)), dim=-1)
    rays_d = (c2w[..., :3, :3] @ dirs.mT).mT
    rays_o = (c2w[..., :3, 3:4].mT).expand(-1, rays_d.shape[1], -1)
    n = torch.norm(rays_d, dim=-1, keepdim=True)
    return rays_o, rays_d / n, n


def bounding_box(c2ws: torch.Tensor, K, near: float, far: float):
    """find_bounding_box (helper.py:109-141): bbox of ray points at depths {near, far+1.5}; the image
    size is re-derived as W=2*K[0,2], H=2*K[1,2] from the (integer) principal point (:114-115).
    Returns (max_bound, min_bound) like the reference."""
    t = torch.tensor([near, far + 1.5], dtype=torch.float64)
    W, H = 2 * K[0, 2], 2 * K[1, 2]
    o, d, _ = get_od(H, W, K, c2ws)
    pts = (o[..., None, :] + d[..., None, :] * t[None, :, None]).reshape(-1, 3)
    return pts.max(0).values.to(torch.float32), pts.min(0).values.to(torch.float32)


# ------------------------------------------------------------------------------------------------
# a13/a14: density grid + marching cubes invariants
# ------------------------------------------------------------------------------------------------
def grid_points(min_bound: np.ndarray, max_bound: np.ndarray, res: int) -> torch.Tensor:
    """nerf2mesh.py:31-40: np.linspace per axis, np.meshgrid default 'xy' indexing so that flat index
    p = (i*res + j)*res + k  <->  (x[j], y[i], z[k]); float64 -> float16 positions."""
    x = np.linspace(min_bound[0], max_bound[0], res)
    y = np.linspace(min_bound[1], max_bound[1], res)
    z = np.linspace(min_bound[2], max_bound[2], res)
    X, Y, Z = np.meshgrid(x, y, z)
    g = torch.stack([torch.tensor(X.reshape(-1)), torch.tensor(Y.reshape(-1)), torch.tensor(Z.reshape(-1))], dim=1)
    return g.to(torch.float16)


def grid_query(p_mlp, tables, mu, sigma, scales, pts_f16: torch.Tensor, num_freq=4, batch=400000) -> torch.Tensor:
    """nerf2mesh.py:69-85: fp16 positions, view dir (0,0,1) fp16, fp32 encoder + MLP, batches of 400000.
    Returns (P,4) [rgb, density] fp32."""
    outs = []
    vd = torch.zeros(1, 3, dtype=torch.float16)
    vd[..., 2] = 1.0
    enc_dir = dir_encode(vd, num_freq)                       # fp16 values, promoted by cat in the MLP
    for s in range(0, pts_f16.shape[0], batch):
        x = pts_f16[s:s + batch]
        f = hash_encode(x, tables, mu, sigma, scales)
        outs.append(mlp_forward(p_mlp, f, enc_dir.expand(x.shape[0], -1)))
    return torch.cat(outs, 0)


def mc_crossing_edges(density: np.ndarray, iso: float, i_begin: int = 0, i_end: Optional[int] = None) -> int:
    """Number of grid edges whose endpoints straddle the iso level with the inside test d < iso.
    Equals the vertex count of any table-based marching cubes that welds one vertex per edge.
    With a slab [i_begin, i_end) of axis 0: only edges OWNED by the slab's grid points (an edge belongs to its lower
    end point), the ownership rule of hbr_mc_count -- the slab counts of a partition add up to the whole grid's."""
    inside = density < iso
    n0 = inside.shape[0]
    i_end = n0 if i_end is None else i_end
    own = inside[i_begin:i_end]
    n = 0
    up = inside[i_begin + 1:min(i_end + 1, n0)]                       # axis-0 edges: lower end point i in the slab
    n += int(np.count_nonzero(up != own[:up.shape[0]]))
    n += int(np.count_nonzero(own[:, 1:, :] != own[:, :-1, :]))
    n += int(np.count_nonzero(own[:, :, 1:] != own[:, :, :-1]))
    return n


def mc_case_index(density: np.ndarray, iso: float) -> np.ndarray:
    """8-bit cube configuration per cell; bit v set iff corner v is inside (d < iso), corner order
    v = dx + 2*dy + 4*dz over grid axes (0,1,2).  Shape (n0-1, n1-1, n2-1) uint8."""
    ins = (density < iso)
    idx = np.zeros(tuple(s - 1 for s in density.shape), dtype=np.uint8)
    for v in range(8):
        dx, dy, dz = v & 1, (v >> 1) & 1, (v >> 2) & 1
        sl = ins[dx:dx + density.shape[0] - 1, dy:dy + density.shape[1] - 1, dz:dz + density.shape[2] - 1]
        idx |= (sl.astype(np.uint8) << v)
    return idx


# ------------------------------------------------------------------------------------------------
# bf16 tensor-core numerics of MLP_3D, emulated in torch (checker for csrc/mlp_tc.cu)
# ------------------------------------------------------------------------------------------------
def mlp_tc_emulation(p: Dict[str, torch.Tensor], feat: torch.Tensor, dirs: torch.Tensor, dout: Optional[torch.Tensor] = None,
                     fmt: torch.dtype = torch.bfloat16):

    """MLP_3D forward (and backward when dout is given) with the tensor-core kernel's rounding points:
    weights, layer inputs and pre-activation gradients rounded to the operand format `fmt` (bfloat16 or float16), products/accumulation/bias/activations in
    fp32, the layer-3 vector (density + 15 features) and the outputs NOT rounded.  Returns out (N,4) and, with
    dout, (dfeat, grads dict).  Not a reference restatement -- a numerics model of our own kernel, used to test it
    tightly; the reference-facing tolerance (1e-2, BASELINE.json) is checked against mlp_forward."""
    def _bf(x: torch.Tensor) -> torch.Tensor:
        return x.to(fmt).to(torch.float32)

    # the bias enters the accumulator through the tensor core as bf16(b) + bf16(b - bf16(b))
    W = {k: _bf(v) if k.endswith("weight") else _bf(v) + _bf(v - _bf(v)) for k, v in p.items()}
    x0 = _bf(feat)
    h1p = x0 @ W["sig_model.0.weight"].T + W["sig_model.0.bias"]
    h1 = _bf(torch.relu(h1p))
    h2p = h1 @ W["sig_model.2.weight"].T + W["sig_model.2.bias"]
    h2 = _bf(torch.relu(h2p))
    o = h2 @ W["sig_model.4.weight"].T + W["sig_model.4.bias"]
    cin = _bf(torch.cat((o[:, 1:], dirs), dim=-1))
    c1p = cin @ W["col_model.0.weight"].T + W["col_model.0.bias"]
    c1 = _bf(torch.relu(c1p))
    c2p = c1 @ W["col_model.2.weight"].T + W["col_model.2.bias"]
    c2 = _bf(torch.relu(c2p))
    pre = c2 @ W["col_model.4.weight"].T + W["col_model.4.bias"]
    out = torch.cat((Fnn.elu(pre), Fnn.leaky_relu(o[:, 0:1], 0.01)), dim=-1)
    if dout is None:
        return out
    g = {}
    dz6 = _bf(dout[:, :3] * torch.where(pre > 0, torch.ones_like(pre), torch.exp(pre)))
    g["col_model.4.weight"], g["col_model.4.bias"] = dz6.T @ c2, dz6.sum(0)
    dz5 = _bf((dz6 @ W["col_model.4.weight"]) * (c2p > 0))
    g["col_model.2.weight"], g["col_model.2.bias"] = dz5.T @ c1, dz5.sum(0)
    dz4 = _bf((dz5 @ W["col_model.2.weight"]) * (c1p > 0))
    g["col_model.0.weight"], g["col_model.0.bias"] = dz4.T @ cin, dz4.sum(0)
    dcin = dz4 @ W["col_model.0.weight"]
    d_o = torch.cat((dout[:, 3:4] * torch.where(o[:, 0:1] > 0, 1.0, 0.01), dcin[:, :15]), dim=-1)
    dz3 = _bf(d_o)
    g["sig_model.4.weight"], g["sig_model.4.bias"] = dz3.T @ h2, dz3.sum(0)
    dz2 = _bf((dz3 @ W["sig_model.4.weight"]) * (h2p > 0))
    g["sig_model.2.weight"], g["sig_model.2.bias"] = dz2.T @ h1, dz2.sum(0)
    dz1 = _bf((dz2 @ W["sig_model.2.weight"]) * (h1p > 0))
    g["sig_model.0.weight"], g["sig_model.0.bias"] = dz1.T @ x0, dz1.sum(0)
    dfeat = dz1 @ W["sig_model.0.weight"]
    return out, dfeat, g, dcin[:, 15:]


def mlp_bf16_emulation(p, feat, dirs, dout=None):
    return mlp_tc_emulation(p, feat, dirs, dout, torch.bfloat16)
