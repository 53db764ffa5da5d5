"""Tensor-level wrappers over the C ABI (include/hbr.h) and the autograd glue.

Everything here takes CUDA tensors and raises on anything else -- there is no CPU path.
The wrappers allocate outputs/scratch with torch (caching allocator, current stream) and pass raw
pointers; the native library never allocates.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
HAS_TC = True    # csrc/mlp_tc.cu (tcgen05) is linked in

from ._lib import HBR_BF16, HBR_F16, HBR_F32, HashGeom, MlpDims, check, lib, ptr, require_cuda, stream


# ------------------------------------------------------------------------------------------------------
# geometry helpers
# ------------------------------------------------------------------------------------------------------
def make_geom(mu, sigma, scales: Sequence[float], L: int, F: int, T: int, E: int = 0) -> HashGeom:
    g = HashGeom()
    for i in range(3):
        g.mu[i] = float(mu[i])
    g.sigma = float(sigma)
    g.L, g.F, g.E, g.T = int(L), int(F), int(E), int(T)
    for i in range(L):
        g.scale[i] = float(scales[i])
    return g


def _xdtype(x: torch.Tensor) -> int:
    if x.dtype == torch.float32:
        return HBR_F32
    if x.dtype == torch.float16:
        return HBR_F16
    raise TypeError(f"positions must be float32 or float16, got {x.dtype}")


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ------------------------------------------------------------------------------------------------------
# hash grid
# ------------------------------------------------------------------------------------------------------
def hash_encode_fwd(x: torch.Tensor, table: torch.Tensor, geom: HashGeom) -> torch.Tensor:
    require_cuda(x, table)
    x = x.contiguous()
    n = x.shape[0]
    cols = geom.L * geom.F + geom.E
    y = torch.empty((n, cols), device=x.device, dtype=torch.float32)
    check(lib().hbr_hash_encode_fwd(ptr(x), _xdtype(x), n, ptr(table), C.byref(geom), ptr(y), cols, stream()))
    return y


def hash_encode_bwd(x: torch.Tensor, dy: torch.Tensor, geom: HashGeom, dtable: torch.Tensor, level_begin: int = 0,
                    level_end: Optional[int] = None) -> None:
    """dtable (L,T,F) fp32 is accumulated into; only levels [level_begin, level_end) are processed."""
    require_cuda(x, dy, dtable)
    x = x.contiguous()
    dy = _f32c(dy)
    level_end = geom.L if level_end is None else level_end
    check(lib().hbr_hash_encode_bwd(ptr(x), _xdtype(x), x.shape[0], ptr(dy), dy.stride(0), C.byref(geom), ptr(dtable),
                                    int(level_begin), int(level_end), stream()))


def hash_encode_dx(x: torch.Tensor, table: torch.Tensor, geom: HashGeom, dy: torch.Tensor) -> torch.Tensor:
    """dL/dx (n,3) fp32 for the feature gradient dy (n, >= L*F; columns past L*F are ignored).  Overwritten, not accumulated."""
    require_cuda(x, table, dy)
    x = x.contiguous()
    if dy.dtype != torch.float32 or dy.stride(1) != 1:
        dy = dy.float().contiguous()
    n = x.shape[0]
    dx = torch.empty((n, 3), device=x.device, dtype=torch.float32)
    check(lib().hbr_hash_encode_dx(ptr(x), _xdtype(x), n, ptr(table), C.byref(geom), ptr(dy), dy.stride(0), ptr(dx), stream()))
    return dx


def _t_stride(t: torch.Tensor, S: int) -> int:
    return 0 if t.dim() == 1 else S


_TORCH_OF = {HBR_F32: torch.float32, HBR_F16: torch.float16, HBR_BF16: torch.bfloat16}


def hash_encode_fwd_rays(rays_o, rays_d, t, table, geom: HashGeom, y_dtype: int = HBR_F32) -> torch.Tensor:
    """Encoder forward with the sample positions o + d t formed in the kernel; y (R*S, L*F+E) in fp32 or already rounded to
    the MLP's 16-bit operand format (y_dtype = HBR_F16 | HBR_BF16)."""
    require_cuda(rays_o, rays_d, t, table)
    R, S = rays_o.shape[0], t.shape[-1]
    cols = geom.L * geom.F + geom.E
    y = torch.empty((R * S, cols), device=table.device, dtype=_TORCH_OF[y_dtype])
    check(lib().hbr_hash_encode_fwd_rays(ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, ptr(table), C.byref(geom), ptr(y),
                                         cols, y_dtype, stream()))
    return y


def hash_encode_bwd_rays(rays_o, rays_d, t, dy, geom: HashGeom, dtable, level_begin: int = 0, level_end: Optional[int] = None):
    require_cuda(rays_o, rays_d, t, dy, dtable)
    R, S = rays_o.shape[0], t.shape[-1]
    level_end = geom.L if level_end is None else level_end
    check(lib().hbr_hash_encode_bwd_rays(ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, ptr(dy), dy.stride(0),
                                         C.byref(geom), ptr(dtable), int(level_begin), int(level_end), stream()))


def _bounds(chunks, L):
    b = [int(chunks[0][0])] + [int(c[1]) for c in chunks]
    if (b[0] != 0 or b[-1] != L or any(b[i] >= b[i + 1] for i in range(len(b) - 1))
            or any(int(chunks[i][0]) != int(chunks[i - 1][1]) for i in range(1, len(chunks)))):
        raise ValueError(f"level chunks {chunks} do not partition [0, {L})")
    return (C.c_int * len(b))(*b), len(b) - 1


def hash_bwd_stream_tiles(n_points: int) -> int:
    """CTAs per level chunk of the streamed scatter-add = the count a chunk's `done` word reaches when it is complete."""
    return int(lib().hbr_hash_bwd_stream_tiles(int(n_points)))


def hash_encode_bwd_stream(x, dy, geom: HashGeom, dtable, chunks, done):
    """hash_encode_bwd over all levels in ONE launch that finishes the level chunks [(l0, l1), ...] in order and counts
    finished CTAs per chunk into `done` (int32 device tensor, zeroed by the caller): the producer side of the streamed
    gradient exchange (peer.PeerRegion.all_reduce_stream)."""
    require_cuda(x, dy, dtable, done)
    x = x.contiguous()
    dy = _f32c(dy)
    b, nch = _bounds(chunks, geom.L)
    check(lib().hbr_hash_encode_bwd_stream(ptr(x), _xdtype(x), x.shape[0], ptr(dy), dy.stride(0), C.byref(geom), ptr(dtable),
                                           b, nch, ptr(done), stream()))


def hash_encode_bwd_rays_stream(rays_o, rays_d, t, dy, geom: HashGeom, dtable, chunks, done):
    require_cuda(rays_o, rays_d, t, dy, dtable, done)
    R, S = rays_o.shape[0], t.shape[-1]
    b, nch = _bounds(chunks, geom.L)
    check(lib().hbr_hash_encode_bwd_rays_stream(ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, ptr(dy), dy.stride(0),
                                                C.byref(geom), ptr(dtable), b, nch, ptr(done), stream()))


def hash_bwd_lm_ctas(n_points: int) -> int:
    """CTAs of the level-major scatter-add = the count a chunk's `done` word reaches when the chunk is complete."""
    return int(lib().hbr_hash_bwd_lm_ctas(int(n_points)))


def hash_encode_bwd_lm(x, dy_lm, geom: HashGeom, dtable, chunks=None, done=None):
    """Scatter-add from LEVEL-MAJOR d(features) dy_lm (L, N, F) (mlp_bwd_tc(..., level_major=True)): a co-resident grid
    walks the levels in order, so the table gradient is finished level by level; with chunks = [(l0, l1), ...] and `done`
    (int32 device tensor, zeroed by the caller) every CTA counts itself into done[c] when it has finished chunk c."""
    require_cuda(x, dy_lm, dtable)
    x = x.contiguous()
    assert dy_lm.is_contiguous() and dy_lm.dtype == torch.float32 and dy_lm.shape == (geom.L, x.shape[0], geom.F)
    b, nch = _bounds(chunks, geom.L) if chunks is not None else (None, 0)
    check(lib().hbr_hash_encode_bwd_lm(ptr(x), _xdtype(x), x.shape[0], ptr(dy_lm), C.byref(geom), ptr(dtable), b, nch,
                                       ptr(done), stream()))


def hash_encode_bwd_rays_lm(rays_o, rays_d, t, dy_lm, geom: HashGeom, dtable, chunks=None, done=None):
    require_cuda(rays_o, rays_d, t, dy_lm, dtable)
    R, S = rays_o.shape[0], t.shape[-1]
    assert dy_lm.is_contiguous() and dy_lm.dtype == torch.float32 and dy_lm.shape == (geom.L, R * S, geom.F)
    b, nch = _bounds(chunks, geom.L) if chunks is not None else (None, 0)
    check(lib().hbr_hash_encode_bwd_rays_lm(ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, ptr(dy_lm), C.byref(geom),
                                            ptr(dtable), b, nch, ptr(done), stream()))


def occupancy_update(pts, alpha, grid, mu, sigma: float, flags2):
    """Volume_Renderer.update_grid (vol_renderer.py:116-131) in place on `grid` ((G,G,G) bool)."""
    require_cuda(pts, alpha, grid, flags2)
    pts = _f32c(pts.reshape(-1, 3))
    alpha = _f32c(alpha.reshape(-1))
    mu3 = (C.c_float * 3)(*[float(v) for v in mu])
    check(lib().hbr_occupancy_update(ptr(pts), pts.shape[0], ptr(alpha), 1, ptr(grid), grid.shape[0], mu3, float(sigma),
                                     ptr(flags2), stream()))


def compact_samples(rays_o, rays_d, t, grid, mu, sigma: float):
    """Live samples of the rays under the occupancy grid: (pts_c (R*S,3), ray_c (R*S) int32, rowmap (R*S) int32,
    count (1) uint64 on the device); only the first `count` rows of pts_c / ray_c are meaningful."""
    require_cuda(rays_o, rays_d, t, grid)
    R, S = rays_o.shape[0], t.shape[-1]
    dev = rays_o.device
    pts_c = torch.empty((R * S, 3), device=dev, dtype=torch.float32)
    ray_c = torch.empty((R * S,), device=dev, dtype=torch.int32)
    rowmap = torch.empty((R * S,), device=dev, dtype=torch.int32)
    count = torch.zeros(1, device=dev, dtype=torch.int64)
    mu3 = (C.c_float * 3)(*[float(v) for v in mu])
    check(lib().hbr_compact_samples(ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, ptr(grid), grid.shape[0], mu3,
                                    float(sigma), ptr(pts_c), ptr(ray_c), ptr(rowmap), ptr(count), stream()))
    return pts_c, ray_c, rowmap, count


def hash_encode_fwd_pts(x, n_dev, table, geom: HashGeom, y_dtype: int = HBR_F32) -> torch.Tensor:
    require_cuda(x, table)
    n = x.shape[0]
    cols = geom.L * geom.F + geom.E
    y = torch.empty((n, cols), device=table.device, dtype=_TORCH_OF[y_dtype])
    check(lib().hbr_hash_encode_fwd_pts(ptr(x), n, ptr(n_dev), ptr(table), C.byref(geom), ptr(y), cols, y_dtype, stream()))
    return y


def hash_encode_bwd_pts(x, n_dev, dy, geom: HashGeom, dtable, level_begin: int = 0, level_end: Optional[int] = None):
    require_cuda(x, dy, dtable)
    level_end = geom.L if level_end is None else level_end
    check(lib().hbr_hash_encode_bwd_pts(ptr(x), x.shape[0], ptr(n_dev), ptr(dy), dy.stride(0), C.byref(geom), ptr(dtable),
                                        int(level_begin), int(level_end), stream()))


def hash_indices(x: torch.Tensor, geom: HashGeom, want_w: bool = True):
    require_cuda(x)
    x = x.contiguous()
    n = x.shape[0]
    idx = torch.empty((geom.L, n, 8), device=x.device, dtype=torch.int32)
    w = torch.empty((geom.L, n, 8), device=x.device, dtype=torch.float32) if want_w else None
    check(lib().hbr_hash_indices(ptr(x), _xdtype(x), n, C.byref(geom), ptr(idx), ptr(w), stream()))
    return idx, w


# ------------------------------------------------------------------------------------------------------
# direction encoding, sample positions, occupancy
# ------------------------------------------------------------------------------------------------------
def dir_encode(d: torch.Tensor, num_freq: int) -> torch.Tensor:
    require_cuda(d)
    d = d.contiguous()
    n, dim = d.shape
    out = torch.empty((n, dim * 2 * num_freq), device=d.device, dtype=torch.float32)
    check(lib().hbr_dir_encode(ptr(d), _xdtype(d), n, dim, num_freq, ptr(out), stream()))
    return out


def ray_points(rays_o: torch.Tensor, rays_d: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    require_cuda(rays_o, rays_d, t)
    rays_o, rays_d, t = _f32c(rays_o), _f32c(rays_d), _f32c(t)
    R = rays_o.shape[0]
    S = t.shape[-1]
    pts = torch.empty((R, S, 3), device=rays_o.device, dtype=torch.float32)
    check(lib().hbr_ray_points(ptr(rays_o), ptr(rays_d), ptr(t), 0 if t.dim() == 1 else S, R, S, ptr(pts), stream()))
    return pts


def _intrinsics(K) -> tuple:
    """(fx, fy, cx, cy) as Python floats from the reference's 3x3 K (int64 at train_hash2.py:67-72, any dtype here)."""
    K = torch.as_tensor(K).detach().cpu()
    return float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])


def ray_gen(c2w: torch.Tensor, H: int, W: int, K, ray_ids: Optional[torch.Tensor] = None, first: int = 0,
            n_rays: Optional[int] = None, images: Optional[torch.Tensor] = None, check_ids: bool = False):
    """helper.py:176-208 per requested ray (id = view*H*W + row*W + col).  c2w (V,4,4) fp32 CUDA; images (V,H,W,3)
    fp32 or uint8.  Returns rays_o (n,3), rays_d (n,3), dir_norm (n,1), gt (n,3) or None."""
    require_cuda(c2w, ray_ids, images)
    c2w = c2w.float().contiguous()
    V = c2w.shape[0]
    if c2w.shape[1:] != (4, 4):
        raise ValueError("c2w must be (V,4,4)")
    if ray_ids is not None:
        ray_ids = ray_ids.to(torch.int64).contiguous()
        n_rays = ray_ids.numel()
    elif n_rays is None:
        n_rays = V * H * W - first
    dtype = HBR_F32
    if images is not None:
        if tuple(images.shape) != (V, H, W, 3) or not images.is_contiguous():
            raise ValueError("images must be contiguous (V,H,W,3)")
        if images.dtype == torch.uint8:
            dtype = _lib.HBR_U8
        elif images.dtype != torch.float32:
            raise TypeError("images must be float32 or uint8")
    dev = c2w.device
    o = torch.empty((n_rays, 3), device=dev)
    d = torch.empty((n_rays, 3), device=dev)
    nrm = torch.empty((n_rays, 1), device=dev)
    gt = torch.empty((n_rays, 3), device=dev) if images is not None else None
    bad = torch.zeros(1, dtype=torch.int32, device=dev) if check_ids else None
    fx, fy, cx, cy = _intrinsics(K)
    check(lib().hbr_ray_gen(ptr(c2w), V, int(H), int(W), fx, fy, cx, cy, ptr(ray_ids), int(first), int(n_rays), ptr(images), dtype,
                            ptr(o), ptr(d), ptr(nrm), ptr(gt), ptr(bad), stream()))
    if check_ids and int(bad.item()):
        raise IndexError("ray id outside [0, V*H*W)")
    return o, d, nrm, gt


def ray_bbox(c2w: torch.Tensor, H: int, W: int, K, t0: float, t1: float, bounds: Optional[torch.Tensor] = None) -> torch.Tensor:
    """helper.py:109-141 over the views in c2w: updates / returns bounds = [min xyz, max xyz] (6 floats on the device)."""
    require_cuda(c2w, bounds)
    c2w = c2w.float().contiguous()
    if bounds is None:
        bounds = torch.tensor([1e7, 1e7, 1e7, -1e7, -1e7, -1e7], device=c2w.device)
    fx, fy, cx, cy = _intrinsics(K)
    check(lib().hbr_ray_bbox(ptr(c2w), c2w.shape[0], int(H), int(W), fx, fy, cx, cy, float(t0), float(t1), ptr(bounds), stream()))
    return bounds


def occupancy_mask(pts: torch.Tensor, grid: torch.Tensor, mu, sigma: float) -> torch.Tensor:
    require_cuda(pts, grid)
    pts = _f32c(pts)
    n = pts.numel() // 3
    mask = torch.empty(pts.shape[:-1], device=pts.device, dtype=torch.bool)
    mu3 = (C.c_float * 3)(*[float(v) for v in mu])
    check(lib().hbr_occupancy_mask(ptr(pts), n, ptr(grid), grid.shape[0], mu3, float(sigma), ptr(mask), stream()))
    return mask


# ------------------------------------------------------------------------------------------------------
# compositing / hierarchical sampling
# ------------------------------------------------------------------------------------------------------
def _dn_args(dir_norm, R, device):
    if torch.is_tensor(dir_norm):
        if dir_norm.numel() == 1:
            return None, float(dir_norm)
        dn = _f32c(dir_norm.reshape(-1))
        if dn.shape[0] != R:
            raise ValueError(f"dir_norm has {dn.shape[0]} rows, expected {R}")
        return dn.to(device), 1.0
    return None, float(dir_norm)


ERT_TAU = 104.0       # exp(-104) == 0 in fp32: the transmittance of every sample skipped by early ray termination is exactly 0


def composite_fwd(t, rgb, rgb_stride, sigma, sigma_stride, dir_norm, mask, R, S, want_w=True, ert_tau=0.0, rowmap=None):
    dn, dns = _dn_args(dir_norm, R, t.device)
    Cc = torch.empty((R, 3), device=t.device, dtype=torch.float32)
    w = torch.empty((R, S), device=t.device, dtype=torch.float32) if want_w else None
    check(lib().hbr_composite_fwd(ptr(t), 0 if t.dim() == 1 else S, ptr(rgb), rgb_stride, ptr(sigma), sigma_stride,
                                  ptr(dn), dns, ptr(mask), ptr(rowmap), R, S, ptr(Cc), ptr(w), float(ert_tau), stream()))
    return Cc, w


def composite_bwd(t, rgb, rgb_stride, sigma, sigma_stride, dir_norm, mask, R, S, gC, drgb, drgb_stride, dsig, dsig_stride,
                  ert_tau=0.0, rowmap=None):
    dn, dns = _dn_args(dir_norm, R, t.device)
    check(lib().hbr_composite_bwd(ptr(t), 0 if t.dim() == 1 else S, ptr(rgb), rgb_stride, ptr(sigma), sigma_stride,
                                  ptr(dn), dns, ptr(mask), ptr(rowmap), R, S, ptr(gC), ptr(drgb), drgb_stride, ptr(dsig), dsig_stride,
                                  float(ert_tau), stream()))


def composite_maps_fwd(t, rgb, rgb_stride, sigma, sigma_stride, dir_norm, mask, R, S, want_w=True, ert_tau=0.0, rowmap=None,
                       want_depth=True, want_opacity=True):
    """composite_fwd plus the per-ray maps depth = sum w t (units of t; z-depth = depth / dir_norm) and opacity = sum w, in
    the same kernel.  Returns (C (R,3), w (R,S) or None, depth (R) or None, opacity (R) or None)."""
    dn, dns = _dn_args(dir_norm, R, t.device)
    Cc = torch.empty((R, 3), device=t.device, dtype=torch.float32)
    w = torch.empty((R, S), device=t.device, dtype=torch.float32) if want_w else None
    D = torch.empty((R,), device=t.device, dtype=torch.float32) if want_depth else None
    A = torch.empty((R,), device=t.device, dtype=torch.float32) if want_opacity else None
    check(lib().hbr_composite_maps_fwd(ptr(t), 0 if t.dim() == 1 else S, ptr(rgb), rgb_stride, ptr(sigma), sigma_stride,
                                       ptr(dn), dns, ptr(mask), ptr(rowmap), R, S, ptr(Cc), ptr(w), ptr(D), ptr(A),
                                       float(ert_tau), stream()))
    return Cc, w, D, A


def composite_maps_bwd(t, rgb, rgb_stride, sigma, sigma_stride, dir_norm, mask, R, S, gC, gD, gA, drgb, drgb_stride, dsig,
                       dsig_stride, ert_tau=0.0, rowmap=None):
    """composite_bwd with the gradients gD, gA (R) of the depth and opacity maps; any of gC, gD, gA may be None (= 0)."""
    dn, dns = _dn_args(dir_norm, R, t.device)
    check(lib().hbr_composite_maps_bwd(ptr(t), 0 if t.dim() == 1 else S, ptr(rgb), rgb_stride, ptr(sigma), sigma_stride,
                                       ptr(dn), dns, ptr(mask), ptr(rowmap), R, S, ptr(gC), ptr(gD), ptr(gA), ptr(drgb),
                                       drgb_stride, ptr(dsig), dsig_stride, float(ert_tau), stream()))


class CompositePacked(torch.autograd.Function):
    """calc_color on the MLP's packed (R*S,4) [rgb,sigma] output -> (C (R,3), w (R,S)); w carries no gradient."""

    @staticmethod
    def forward(ctx, out4, t, dir_norm, mask, R, S, ert_tau=0.0, rowmap=None):
        """rowmap (R*S) int32: out4 is a COMPACTED (n_live.., 4) list; sample i lives at row rowmap[i] (< 0: skipped)."""
        require_cuda(out4, t)
        out4 = _f32c(out4)
        t = _f32c(t)
        ctx.ert_tau = float(ert_tau)
        Cc, w = composite_fwd(t, out4, 4, out4[:, 3:], 4, dir_norm, mask, R, S, ert_tau=ert_tau, rowmap=rowmap)
        ctx.rowmap = rowmap
        ctx.save_for_backward(out4, t, dir_norm if torch.is_tensor(dir_norm) else None, mask)
        ctx.dn_scalar = None if torch.is_tensor(dir_norm) else dir_norm
        ctx.RS = (R, S)
        ctx.mark_non_differentiable(w)
        return Cc, w

    @staticmethod
    def backward(ctx, gC, _gw):
        out4, t, dn, mask = ctx.saved_tensors
        dn = dn if dn is not None else ctx.dn_scalar
        R, S = ctx.RS
        d4 = torch.empty_like(out4)
        composite_bwd(t, out4, 4, out4[:, 3:], 4, dn, mask, R, S, _f32c(gC), d4, 4, d4[:, 3:], 4, ert_tau=ctx.ert_tau,
                      rowmap=ctx.rowmap)
        return d4, None, None, None, None, None, None, None


class CompositeMapsPacked(torch.autograd.Function):
    """CompositePacked with the depth and opacity maps: out4 (R*S,4) [rgb, sigma] (or a compacted list read through rowmap)
    -> (C (R,3), w (R,S), depth (R), opacity (R)).  C, depth and opacity carry gradients, w does not.  depth = sum_s w_s t_s
    is the distance along the unit ray direction (z-depth = depth / dir_norm), opacity = sum_s w_s; neither is normalised
    or clamped."""

    @staticmethod
    def forward(ctx, out4, t, dir_norm, mask, R, S, ert_tau=0.0, rowmap=None):
        require_cuda(out4, t)
        out4 = _f32c(out4)
        t = _f32c(t)
        ctx.ert_tau = float(ert_tau)
        Cc, w, D, A = composite_maps_fwd(t, out4, 4, out4[:, 3:], 4, dir_norm, mask, R, S, ert_tau=ert_tau, rowmap=rowmap)
        ctx.rowmap = rowmap
        ctx.save_for_backward(out4, t, dir_norm if torch.is_tensor(dir_norm) else None, mask)
        ctx.dn_scalar = None if torch.is_tensor(dir_norm) else dir_norm
        ctx.RS = (R, S)
        ctx.mark_non_differentiable(w)
        ctx.set_materialize_grads(False)          # an unused map costs no zero-filled gradient: the kernel reads NULL as 0
        return Cc, w, D, A

    @staticmethod
    def backward(ctx, gC, _gw, gD, gA):
        if gC is None and gD is None and gA is None:
            return (None,) * 8
        out4, t, dn, mask = ctx.saved_tensors
        dn = dn if dn is not None else ctx.dn_scalar
        R, S = ctx.RS
        d4 = torch.empty_like(out4)
        composite_maps_bwd(t, out4, 4, out4[:, 3:], 4, dn, mask, R, S, _f32c(gC), _f32c(gD), _f32c(gA), d4, 4, d4[:, 3:], 4,
                           ert_tau=ctx.ert_tau, rowmap=ctx.rowmap)
        return d4, None, None, None, None, None, None, None


class CompositeSplit(torch.autograd.Function):
    """calc_color on separate rgb (R,S,3) / sigma (R,S) tensors (the free-function API of helper.py)."""

    @staticmethod
    def forward(ctx, rgb, sigma, t, dir_norm, mask):
        require_cuda(rgb, sigma, t)
        rgb, sigma, t = _f32c(rgb), _f32c(sigma), _f32c(t)
        R, S = sigma.shape
        Cc, w = composite_fwd(t, rgb, 3, sigma, 1, dir_norm, mask, R, S)
        ctx.save_for_backward(rgb, sigma, t, dir_norm if torch.is_tensor(dir_norm) else None, mask)
        ctx.dn_scalar = None if torch.is_tensor(dir_norm) else dir_norm
        ctx.mark_non_differentiable(w)
        return Cc, w

    @staticmethod
    def backward(ctx, gC, _gw):
        rgb, sigma, t, dn, mask = ctx.saved_tensors
        dn = dn if dn is not None else ctx.dn_scalar
        R, S = sigma.shape
        drgb = torch.empty_like(rgb)
        dsig = torch.empty_like(sigma)
        composite_bwd(t, rgb, 3, sigma, 1, dn, mask, R, S, _f32c(gC), drgb, 3, dsig, 1)
        return drgb, dsig, None, None, None


# ------------------------------------------------------------------------------------------------------
# SDF mode (SURVEY 8f row 4): csrc/sdf.cu
# ------------------------------------------------------------------------------------------------------
def _sample_stride(x: torch.Tensor, width: int) -> Optional[int]:
    """Element stride between consecutive samples of an (R,S[,width]) tensor whose samples are uniformly strided (a
    contiguous tensor, or a column view of the MLP's packed (R*S,4) output); None if it has to be copied."""
    R, S = x.shape[0], x.shape[1]
    if x.dim() == 3 and (x.shape[2] != width or (width > 1 and x.stride(2) != 1)):
        return None
    st = x.stride(1) if S > 1 else (x.stride(0) if R > 1 else max(width, 1))
    if R > 1 and x.stride(0) != S * st:
        return None
    return int(st) if st >= width else None


def _sdf_views(rgb, sdf):
    if rgb.dtype != torch.float32 or _sample_stride(rgb, 3) is None:
        rgb = rgb.float().contiguous()
    if sdf.dtype != torch.float32 or _sample_stride(sdf, 1) is None:
        sdf = sdf.float().contiguous()
    return rgb, _sample_stride(rgb, 3), sdf, _sample_stride(sdf, 1)


def _composite_sdf_fwd(rgb, rgb_st, sdf, sdf_st, from_density, b32, R, S):
    Cc = torch.empty((R, 3), device=sdf.device, dtype=torch.float32)
    w = torch.empty((R, S), device=sdf.device, dtype=torch.float32)
    check(lib().hbr_composite_sdf_fwd(ptr(rgb), rgb_st, ptr(sdf), sdf_st, from_density, ptr(b32), R, S, ptr(Cc), ptr(w), stream()))
    return Cc, w


def _composite_sdf_bwd(rgb, rgb_st, sdf, sdf_st, from_density, b32, R, S, gC, gw):
    """-> (d4 (R*S,4) packed [d rgb, d sdf] (one 16-byte store per sample), dL/db as a 0-dim tensor)."""
    dev = b32.device
    d4 = torch.empty((R * S, 4), device=dev, dtype=torch.float32)
    db_ray = torch.empty((R,), device=dev, dtype=torch.float32)
    gC = _f32c(gC) if gC is not None else torch.zeros((R, 3), device=dev)
    gw = _f32c(gw.reshape(R, S)) if gw is not None else None
    check(lib().hbr_composite_sdf_bwd(ptr(rgb), rgb_st, ptr(sdf), sdf_st, from_density, ptr(b32), R, S, ptr(gC), ptr(gw),
                                      ptr(d4), 4, ptr(d4[:, 3:]), 4, ptr(db_ray), stream()))
    return d4, db_ray.sum()


class CompositeSdf(torch.autograd.Function):
    """calc_color's SDF branch (helper.py:76-86,102-105) on rgb (R,S,3) / sdf (R,S) with VarModel's sharpness b (0-dim
    parameter) -> (C (R,3), w (R,S)).  from_density: `sdf` holds the density head's LeakyReLU output and the SDF value
    2*sigmoid(pre-activation) - 1 (test_hash.py:59-60) is formed inside the kernel."""

    @staticmethod
    def forward(ctx, rgb, sdf, b, from_density=False):
        require_cuda(rgb, sdf, b)
        R, S = sdf.shape
        rgb, rgb_st, sdf, sdf_st = _sdf_views(rgb, sdf)
        b32 = b.detach().reshape(1).float().contiguous()
        Cc, w = _composite_sdf_fwd(rgb, rgb_st, sdf, sdf_st, int(bool(from_density)), b32, R, S)
        ctx.save_for_backward(rgb, sdf, b32)
        ctx.meta = (rgb_st, sdf_st, int(bool(from_density)), b.shape, b.dtype)
        ctx.set_materialize_grads(False)          # an unused weight output costs no zero-filled (R,S) gradient
        return Cc, w

    @staticmethod
    def backward(ctx, gC, gw):
        rgb, sdf, b32 = ctx.saved_tensors
        rgb_st, sdf_st, from_density, b_shape, b_dtype = ctx.meta
        R, S = sdf.shape
        d4, db = _composite_sdf_bwd(rgb, rgb_st, sdf, sdf_st, from_density, b32, R, S, gC, gw)
        d4 = d4.view(R, S, 4)
        return d4[..., :3], d4[..., 3], db.reshape(b_shape).to(b_dtype), None


class CompositeSdfPacked(torch.autograd.Function):
    """The same on the MLP's packed (R*S,4) [rgb, density-or-sdf] output: no column views, the gradient goes back as one
    (R*S,4) tensor (Volume_Renderer's native SDF route)."""

    @staticmethod
    def forward(ctx, out4, b, R, S, from_density=True):
        require_cuda(out4, b)
        out4 = _f32c(out4)
        b32 = b.detach().reshape(1).float().contiguous()
        Cc, w = _composite_sdf_fwd(out4, 4, out4[:, 3:], 4, int(bool(from_density)), b32, R, S)
        ctx.save_for_backward(out4, b32)
        ctx.meta = (R, S, int(bool(from_density)), b.shape, b.dtype)
        ctx.set_materialize_grads(False)
        return Cc, w

    @staticmethod
    def backward(ctx, gC, gw):
        out4, b32 = ctx.saved_tensors
        R, S, from_density, b_shape, b_dtype = ctx.meta
        d4, db = _composite_sdf_bwd(out4, 4, out4[:, 3:], 4, from_density, b32, R, S, gC, gw)
        return d4, db.reshape(b_shape).to(b_dtype), None, None, None


def sdf_stencil_points(x: torch.Tensor, eps: float, lo, hi) -> torch.Tensor:
    """x (n,3) -> (6,n,3): clamp(x +- eps e_axis, lo, hi) for axis = x, y, z (test_hash.py:91-102), slabs [+x, -x, +y, ...]."""
    require_cuda(x)
    x = _f32c(x)
    n = x.shape[0]
    pts = torch.empty((6, n, 3), device=x.device, dtype=torch.float32)
    lo3, hi3 = (C.c_float * 3)(*lo), (C.c_float * 3)(*hi)
    check(lib().hbr_sdf_stencil_points(ptr(x), n, float(eps), lo3, hi3, ptr(pts), stream()))
    return pts


class SdfEikonal(torch.autograd.Function):
    """dens6 (6,n): LeakyReLU density-head output at the stencil points -> (norm (n), grads (n,3)): the central differences
    of 2*sigmoid(pre-activation) - 1 and their Euclidean norm (test_hash.py:104, helper.py:293-297).  Only the norm carries
    a gradient."""

    @staticmethod
    def forward(ctx, dens6, eps):
        require_cuda(dens6)
        dens6 = _f32c(dens6)
        n = dens6.shape[1]
        norm = torch.empty((n,), device=dens6.device, dtype=torch.float32)
        grads = torch.empty((n, 3), device=dens6.device, dtype=torch.float32)
        check(lib().hbr_sdf_eikonal_fwd(ptr(dens6), n, float(eps), ptr(norm), ptr(grads), stream()))
        ctx.save_for_backward(dens6)
        ctx.eps = float(eps)
        ctx.mark_non_differentiable(grads)
        return norm, grads

    @staticmethod
    def backward(ctx, gnorm, _ggrads):
        (dens6,) = ctx.saved_tensors
        n = dens6.shape[1]
        dd = torch.empty_like(dens6)
        check(lib().hbr_sdf_eikonal_bwd(ptr(dens6), n, ctx.eps, ptr(_f32c(gnorm)), ptr(dd), stream()))
        return dd, None


def hier_sample(w: torch.Tensor, t: torch.Tensor, u: torch.Tensor, cand: torch.Tensor, clamp_in_place=False) -> torch.Tensor:
    require_cuda(w, t, u, cand)
    R, S = w.shape
    assert w.dtype == torch.float32 and w.is_contiguous()
    t, u, cand = _f32c(t), _f32c(u), _f32c(cand)
    tf = torch.empty((R, 2 * S), device=w.device, dtype=torch.float32)
    check(lib().hbr_hier_sample(ptr(w), ptr(t), ptr(u), ptr(cand), R, S, 1 if clamp_in_place else 0, ptr(tf), stream()))
    return tf


def strat_depths(lin: torch.Tensor, u: torch.Tensor, span: float, count: float) -> torch.Tensor:
    """helper.py:231-232: lin + (u * span) / count, each operation rounded on its own (one kernel instead of three)."""
    require_cuda(lin, u)
    lin, u = _f32c(lin), _f32c(u)
    t = torch.empty_like(lin)
    check(lib().hbr_strat_depths(ptr(lin), ptr(u), float(span), float(count), lin.numel(), ptr(t), stream()))
    return t


class MsePair(torch.autograd.Function):
    """nn.MSELoss()(a, gt) [+ nn.MSELoss()(b, gt)] (train_hash2.py:177,221) as one kernel per direction."""

    @staticmethod
    def forward(ctx, a, b, gt, scale=1.0):
        require_cuda(a, b, gt)
        a, gt = _f32c(a), _f32c(gt)
        b = _f32c(b) if b is not None else None
        if a.shape != gt.shape or (b is not None and b.shape != gt.shape):
            raise ValueError("MsePair: shapes differ")
        loss = torch.zeros((), device=a.device, dtype=torch.float32)
        check(lib().hbr_mse_pair_fwd(ptr(a), ptr(b), ptr(gt), a.numel(), float(scale), ptr(loss), stream()))
        ctx.save_for_backward(a, b, gt)
        ctx.scale = float(scale)
        return loss

    @staticmethod
    def backward(ctx, gout):
        a, b, gt = ctx.saved_tensors
        da = torch.empty_like(a)
        db = torch.empty_like(b) if b is not None else None
        gout = _f32c(gout)
        check(lib().hbr_mse_pair_bwd(ptr(a), ptr(b), ptr(gt), a.numel(), ctx.scale, ptr(gout), ptr(da), ptr(db), stream()))
        return da, db, None, None


def mse_pair(a: torch.Tensor, b: Optional[torch.Tensor], gt: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """scale * (mse(a, gt) + mse(b, gt)) (b may be None)."""
    return MsePair.apply(a, b, gt, scale)


# ------------------------------------------------------------------------------------------------------
# MLP (fp32 CUDA-core path)
# ------------------------------------------------------------------------------------------------------
def mlp_act_rows() -> int:
    return int(lib().hbr_mlp_act_floats())


def mlp_fwd_f32(feat, dirs, dir_group, params, dims: MlpDims, keep_act: bool):
    require_cuda(feat, params)
    feat = _f32c(feat)
    n = feat.shape[0]
    out = torch.empty((n, 4 if dirs is not None else 1), device=feat.device, dtype=torch.float32)
    act = torch.empty((mlp_act_rows(), n), device=feat.device, dtype=torch.float32) if keep_act else None
    check(lib().hbr_mlp_fwd_f32(ptr(feat), feat.stride(0), ptr(dirs), dir_group, n, ptr(params), C.byref(dims), ptr(out),
                                ptr(act), stream()))
    return out, act


def mlp_bwd_f32(feat, dirs, dir_group, params, dims: MlpDims, dout, act, want_dfeat, want_ddirs, dparams):
    n = feat.shape[0]
    dz = torch.empty_like(act)
    dfeat = torch.empty((n, dims.in0), device=feat.device, dtype=torch.float32) if want_dfeat else None
    ddirs = torch.zeros_like(dirs) if want_ddirs else None
    check(lib().hbr_mlp_bwd_f32(ptr(feat), feat.stride(0), ptr(dirs), dir_group, n, ptr(params), C.byref(dims), ptr(dout),
                                ptr(act), ptr(dz), ptr(dfeat), dims.in0, ptr(ddirs), ptr(dparams), stream()))
    return dfeat, ddirs


_tc_scratch = {}
_tc_image = {}          # id(scratch buffer) -> (params data_ptr, params version, operand): what the operand image was built from


def mlp_tc_scratch(dims: MlpDims, device) -> torch.Tensor:
    """Per-device scratch of the tensor-core MLP kernels (operand image + per-CTA gradient rows), allocated once."""
    key = (torch.device(device).index, dims.in0, dims.d_view)
    buf = _tc_scratch.get(key)
    if buf is None:
        buf = torch.empty(int(lib().hbr_mlp_tc_scratch_bytes(C.byref(dims))), device=device, dtype=torch.uint8)
        _tc_scratch[key] = buf
    return buf


def tc_operand(dtype=None) -> int:
    """Tensor-core operand format of the MLP kernels for an autocast dtype: float16 -> HBR_F16 (the reference trainer's
    precision, train_hash2.py:218), bfloat16 -> HBR_BF16.  None = the active CUDA autocast dtype (bf16 outside autocast)."""
    if dtype is None:
        dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled() else torch.bfloat16
    if isinstance(dtype, int):
        if dtype in (HBR_F16, HBR_BF16):
            return dtype
        raise ValueError(f"operand format {dtype}")
    if dtype == torch.float16:
        return HBR_F16
    if dtype == torch.bfloat16:
        return HBR_BF16
    raise TypeError(f"the tensor-core MLP runs fp16 or bf16 operands, not {dtype}")


def _operand_torch_dtype(operand: int):
    return torch.float16 if operand == HBR_F16 else torch.bfloat16


def _feat_dtype(feat: torch.Tensor, operand: int) -> int:
    """HBR_F32, or the operand format when the features were produced in it already (hash_encode_fwd_rays)."""
    if feat.dtype == torch.float32:
        return HBR_F32
    if feat.dtype == _operand_torch_dtype(operand):
        return operand
    raise TypeError(f"features are {feat.dtype}; the MLP kernels take float32 or their own operand format")


def _image_key(params, operand):
    return (params.data_ptr(), params._version, operand)


def mlp_tc_prepare(params, dims: MlpDims, operand: int):
    """Build the operand image of `params` on the CURRENT stream (callers put it beside the hash-grid kernel on a side stream
    and join before the MLP kernel); the following mlp_fwd_tc(image_ready=True) / mlp_bwd_tc calls reuse it."""
    scratch = mlp_tc_scratch(dims, params.device)
    check(lib().hbr_mlp_tc_prepare(ptr(params), C.byref(dims), operand, ptr(scratch), stream()))
    _tc_image[id(scratch)] = _image_key(params, operand)


def mlp_fwd_tc(feat, dirs, dir_group, params, dims: MlpDims, keep_act: bool = False, operand: int = HBR_BF16,
               image_ready: bool = False, n_dev=None, dir_rows=None, n_max=None):
    """16-bit tensor-core forward; keeps nothing (the backward recomputes), returns (out, None)."""
    require_cuda(feat, dirs, params)
    n = feat.shape[0]
    out = torch.empty((n, 4), device=feat.device, dtype=torch.float32)
    n = n if n_max is None else int(n_max)
    scratch = mlp_tc_scratch(dims, feat.device)
    # unless the caller has just prepared it (mlp_tc_prepare), the forward rebuilds the operand image (4 us) and records
    # what it was built from; the backward of the same parameters (same storage, same version counter, same operand
    # format) skips its prep kernel
    ready = 1 if (image_ready and _tc_image.get(id(scratch)) == _image_key(params, operand)) else 0
    check(lib().hbr_mlp_fwd_tc(ptr(feat), _feat_dtype(feat, operand), feat.stride(0), ptr(dirs), dir_group, n, ptr(params),
                               C.byref(dims), operand, ptr(out), ptr(scratch), ready, ptr(n_dev), ptr(dir_rows), stream()))
    if ready:
        _lib.STATS.launches -= 1
    _tc_image[id(scratch)] = _image_key(params, operand)
    return out, None


def mlp_tc_reduce_grads(dims: MlpDims, n: int, dparams, device):
    """Second half of mlp_bwd_tc(defer_reduce=True): per-CTA gradient rows -> dparams (accumulating), on the current stream."""
    check(lib().hbr_mlp_tc_reduce_grads(C.byref(dims), int(n), ptr(mlp_tc_scratch(dims, device)), ptr(dparams), stream()))


def mlp_bwd_tc(feat, dirs, dir_group, params, dims: MlpDims, out, dout, want_dfeat, want_ddirs, dparams,
               operand: int = HBR_BF16, grad_scale: float = 1.0, defer_reduce: bool = False, n_dev=None, dir_rows=None,
               level_major: bool = False):
    """`out` is the forward output (N,4): the kernel takes ELU' / LeakyReLU' from it instead of recomputing the last layer.
    defer_reduce: leave the per-CTA gradient rows in the scratch; the caller runs mlp_tc_reduce_grads (on any stream that
    waits for this one) before anything else uses the scratch or reads dparams.
    level_major: dfeat comes back as (in0/2, N, 2) -- level-major, for hash_encode_bwd*_lm (see mlp_level_major_ok)."""
    n = feat.shape[0]
    if level_major and want_dfeat:
        dfeat = torch.empty((dims.in0 // 2, n, 2), device=feat.device, dtype=torch.float32)
    else:
        level_major = False
        dfeat = torch.empty((n, dims.in0), device=feat.device, dtype=torch.float32) if want_dfeat else None
    ddirs = torch.zeros_like(dirs) if want_ddirs else None
    scratch = mlp_tc_scratch(dims, feat.device)
    key = _image_key(params, operand)
    ready = 1 if _tc_image.get(id(scratch)) == key else 0
    check(lib().hbr_mlp_bwd_tc(ptr(feat), _feat_dtype(feat, operand), feat.stride(0), ptr(dirs), dir_group, n, ptr(params),
                               C.byref(dims), operand, ptr(out), ptr(dout), ptr(dfeat),
                               _lib.HBR_DFEAT_LEVEL_MAJOR if level_major else dims.in0, ptr(ddirs), ptr(dparams),
                               float(grad_scale), ptr(scratch), ready, 1 if defer_reduce else 0, ptr(n_dev), ptr(dir_rows),
                               stream()))
    _lib.STATS.launches -= ready + (1 if defer_reduce else 0)    # no prep kernel / no reduce kernel in this call
    _tc_image[id(scratch)] = key
    return dfeat, ddirs


def mlp_level_major_ok(geom: HashGeom, dims: MlpDims, n_points: int) -> bool:
    """The reference's configuration family (F = 2, L = 16, E = 0 -> in0 = 32) with an even point count: the MLP backward
    can write d(features) level-major for hash_encode_bwd*_lm."""
    return geom.F == 2 and geom.L == 16 and geom.E == 0 and dims.in0 == 32 and n_points % 2 == 0 and n_points > 0


def field_fwd_tc(x, table, geom: HashGeom, dirs, dir_group, params, dims: MlpDims, operand: int = HBR_BF16):
    """Fused hash-grid encoder + MLP_3D forward (tensor cores).  Returns (out (N,4) fp32, feat16 (N,32) 16-bit = the
    features that were fed to the tensor cores, kept for the backward recompute)."""
    require_cuda(x, table, dirs, params)
    n = x.shape[0]
    out = torch.empty((n, 4), device=x.device, dtype=torch.float32)
    feat16 = torch.empty((n, 32), device=x.device, dtype=_operand_torch_dtype(operand))
    check(lib().hbr_field_fwd_tc(ptr(x), n, ptr(table), C.byref(geom), ptr(dirs), dir_group, ptr(params), C.byref(dims),
                                 operand, ptr(out), ptr(feat16), ptr(mlp_tc_scratch(dims, x.device)), stream()))
    return out, feat16


def field_fwd_rays_tc(rays_o, rays_d, t, table, geom: HashGeom, dirs, params, dims: MlpDims, operand: int = HBR_BF16):
    """hash_encode_fwd_rays + mlp_fwd_tc in ONE kernel (gather warps beside the tile groups, hbr_field_fwd_rays_tc).  Returns
    (out (R*S,4) fp32, feat16 (R*S,32) in the operand format).  Uses the operand image in the scratch when it is current;
    otherwise the kernel converts the parameters itself (it never writes the image: the caller builds it for the backward,
    e.g. on a side stream, with mlp_tc_prepare)."""
    require_cuda(rays_o, rays_d, t, table, dirs, params)
    R, S = rays_o.shape[0], t.shape[-1]
    n = R * S
    out = torch.empty((n, 4), device=table.device, dtype=torch.float32)
    feat16 = torch.empty((n, 32), device=table.device, dtype=_operand_torch_dtype(operand))
    scratch = mlp_tc_scratch(dims, table.device)
    ready = 1 if _tc_image.get(id(scratch)) == _image_key(params, operand) else 0
    check(lib().hbr_field_fwd_rays_tc(ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, ptr(table), C.byref(geom),
                                      ptr(dirs), ptr(params), C.byref(dims), operand, ptr(out), ptr(feat16), ptr(scratch), ready,
                                      stream()))
    return out, feat16


def field_bwd_tc(x, geom: HashGeom, dirs, dir_group, params, dims: MlpDims, feat16, out, dout, dtable, want_ddirs, dparams,
                 operand: int = HBR_BF16, grad_scale: float = 1.0):
    """Fused MLP_3D backward + hash-grid scatter-add: dtable (L,T,2) and dparams are accumulated into."""
    ddirs = torch.zeros_like(dirs) if want_ddirs else None
    check(lib().hbr_field_bwd_tc(ptr(x), x.shape[0], C.byref(geom), ptr(dirs), dir_group, ptr(params), C.byref(dims),
                                 operand, ptr(feat16), ptr(out), ptr(dout), ptr(dtable), ptr(ddirs), ptr(dparams),
                                 float(grad_scale), ptr(mlp_tc_scratch(dims, x.device)), stream()))
    return ddirs


def field_bwd_rays_tc(feat16, rays_o, rays_d, t, geom: HashGeom, dirs, params, dims: MlpDims, out, dout, dtable, want_ddirs,
                      dparams, operand: int = HBR_BF16, grad_scale: float = 1.0, defer_reduce: bool = False):
    """mlp_bwd_tc + hash_encode_bwd_rays in one kernel (scatter warps beside the tile groups): dtable (L,T,2) and dparams are
    accumulated into; returns ddirs or None."""
    require_cuda(feat16, rays_o, rays_d, t, dirs, params, out, dout, dtable)
    R, S = rays_o.shape[0], t.shape[-1]
    ddirs = torch.zeros_like(dirs) if want_ddirs else None
    scratch = mlp_tc_scratch(dims, feat16.device)
    key = _image_key(params, operand)
    ready = 1 if _tc_image.get(id(scratch)) == key else 0
    check(lib().hbr_field_bwd_rays_tc(ptr(feat16), ptr(rays_o), ptr(rays_d), ptr(t), _t_stride(t, S), R, S, C.byref(geom),
                                      ptr(dirs), ptr(params), C.byref(dims), operand, ptr(out), ptr(dout), ptr(dtable),
                                      ptr(ddirs), ptr(dparams), float(grad_scale), ptr(scratch), ready,
                                      1 if defer_reduce else 0, stream()))
    _lib.STATS.launches -= ready + (1 if defer_reduce else 0)
    _tc_image[id(scratch)] = key
    return ddirs


def field_scatter_supported(geom: HashGeom, dims: MlpDims) -> bool:
    """The configuration family hbr_field_bwd_rays_tc covers (the reference's: F = 2, L = 16, power-of-two T, d_view <= 25)."""
    T = int(geom.T)
    return (geom.F == 2 and geom.L == 16 and geom.E == 0 and T >= 2 and (T & (T - 1)) == 0 and dims.in0 == 32
            and dims.d_view + 15 <= 40)


def debug_umma(mode: int, A: torch.Tensor, B: torch.Tensor, M: int, N: int, K: int, operand: int = HBR_BF16) -> torch.Tensor:
    """Self test of the UMMA operand modes (probe library, tests only)."""
    D = torch.empty((M, N), device=A.device, dtype=torch.float32)
    dl = _lib.debug_lib()
    rc = dl.hbr_debug_umma(mode, operand, ptr(A.contiguous()), ptr(B.contiguous()), ptr(D), N, K, stream())
    if rc != 0:
        raise RuntimeError(f"libhbr_b200_debug: {dl.cdll.hbr_last_error().decode()} (status {rc})")
    return D


# ------------------------------------------------------------------------------------------------------
# density grid + marching cubes
# ------------------------------------------------------------------------------------------------------
def grid_points(min_bound, max_bound, res: int, p0: int, count: int, device) -> torch.Tensor:
    mn = (C.c_double * 3)(*[float(v) for v in min_bound])
    mx = (C.c_double * 3)(*[float(v) for v in max_bound])
    pts = torch.empty((count, 3), device=device, dtype=torch.float16)
    with torch.cuda.device(pts.device):
        check(lib().hbr_grid_points(mn, mx, res, p0, count, ptr(pts), stream()))
    return pts


def mlp_density_tf32x3(feat, params, dims: MlpDims):
    """Density head of MLP_3D on (n,32) fp32 features, tensor cores with split-TF32 operands (fp32-level accuracy)."""
    require_cuda(feat, params)
    feat = _f32c(feat)
    out = torch.empty((feat.shape[0],), device=feat.device, dtype=torch.float32)
    check(lib().hbr_mlp_density_tf32x3(ptr(feat), feat.shape[0], ptr(params), C.byref(dims), ptr(out), stream()))
    return out


def grid_density(min_bound, max_bound, res, p0, count, table, geom, params, dims, dir_enc, chunk=1 << 19, cuda_core_mlp=False):
    """chunk: points per pass (default 2^19: the chunk's 64 MB of fp32 features stay in L2 between the encoder and the MLP).
    cuda_core_mlp: force the fp32 CUDA-core MLP (default: the density-only query runs the split-TF32 tensor-core head)."""
    require_cuda(table, params)
    mn = (C.c_double * 3)(*[float(v) for v in min_bound])
    mx = (C.c_double * 3)(*[float(v) for v in max_bound])
    chunk = max(1, min(chunk, count))
    dev = table.device
    out = torch.empty((count, 4) if dir_enc is not None else (count,), device=dev, dtype=torch.float32)
    pts = torch.empty((chunk, 3), device=dev, dtype=torch.float16)
    feat = torch.empty((chunk, dims.in0), device=dev, dtype=torch.float32)
    check(lib().hbr_grid_density(mn, mx, res, p0, count, ptr(table), C.byref(geom), ptr(params), C.byref(dims),
                                 ptr(dir_enc), ptr(out), ptr(pts), ptr(feat), chunk, 1 if cuda_core_mlp else 0, stream()))
    return out


def mc_count(density: torch.Tensor, iso: float, i_begin: int = 0, i_end: Optional[int] = None):
    require_cuda(density)
    density = _f32c(density)
    n0, n1, n2 = density.shape
    i_end = n0 if i_end is None else i_end
    counts = torch.zeros(2, device=density.device, dtype=torch.int64)
    check(lib().hbr_mc_count(ptr(density), n0, n1, n2, float(iso), i_begin, i_end, ptr(counts), stream()))
    return counts


def mc_emit(density: torch.Tensor, iso: float, n_verts: int, n_faces: int):
    require_cuda(density)
    density = _f32c(density)
    n0, n1, n2 = density.shape
    dev = density.device
    edge_id = torch.empty((3, n0, n1, n2), device=dev, dtype=torch.int32)
    verts = torch.empty((max(n_verts, 1), 3), device=dev, dtype=torch.float32)
    faces = torch.empty((max(n_faces, 1), 3), device=dev, dtype=torch.int32)
    cursors = torch.zeros(2, device=dev, dtype=torch.int64)
    check(lib().hbr_mc_emit(ptr(density), n0, n1, n2, float(iso), 0, n0, ptr(edge_id), ptr(verts), n_verts, ptr(faces),
                            n_faces, ptr(cursors), stream()))
    return verts[:n_verts], faces[:n_faces], cursors


def grid_interp(vol: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """vol (C,n0,n1,n2) fp32, pts (n,3) as (x,y,z) = (axis 2, axis 1, axis 0) index coordinates -> (n,C)."""
    require_cuda(vol, pts)
    vol, pts = _f32c(vol), _f32c(pts)
    C_, n0, n1, n2 = vol.shape
    n = pts.shape[0]
    out = torch.empty((n, C_), device=vol.device, dtype=torch.float32)
    check(lib().hbr_grid_interp(ptr(vol), C_, n0, n1, n2, ptr(pts), n, ptr(out), stream()))
    return out
