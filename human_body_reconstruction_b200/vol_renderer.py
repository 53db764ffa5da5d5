"""Drop-in for the reference's vol_renderer.py: `Volume_Renderer` (vol_renderer.py:88-245).

`vol_render(model, rays_d, rays_o, num_samples, t, update_mask, dir_norm, hierarchical) -> (Cr, Cf, norm)`
(note: rays_d BEFORE rays_o, as in the reference).  When the position encoder is the native `HashEncoder`,
the direction encoder the native `PositionalEncoder` and the model the native `MLP_3D` (optionally inside
`nn.DataParallel` on one device), the whole pass runs on the sm_100a kernels: sample positions, occupancy
lookup, hash encode, field MLP (one direction row per RAY instead of the reference's S-fold repeat),
compositing and the hierarchical resampler.  Any other callable falls back to the reference's data flow
(encode -> model(rays[mask], dirs[mask]) -> scatter) with only sampling/compositing on our kernels.
The legacy classic-NeRF MLP class (vol_renderer.py:12-86) is not part of the hot path and is not provided.
"""
from __future__ import annotations

import os
from collections import namedtuple
from typing import Optional, Tuple

import torch
import torch.nn as nn

from . import ops
from .dist import ParamGrad, node_params
from .encoder import PositionalEncoder
from .hash_encoding import HashEncoder
from .helper import calc_color, hierarchical_sampling, strat_sampler
from .test_hash import MLP_3D


class _FieldFn(torch.autograd.Function):
    """Sample positions (N,3) -> (N,4) [rgb, sigma] through the FUSED encoder + MLP kernels (one kernel per direction):
    HashEncoder.forward feeding MLP_3D.forward as vol_renderer.py:179,211 chains them, bf16 tensor-core arithmetic."""

    @staticmethod
    def forward(ctx, pts, dirs, dir_group, enc, mlp, *params):
        geom, dims = enc._geom(), mlp._dims()
        dirs = dirs.float().contiguous()
        operand = ops.tc_operand()
        out, feat16 = ops.field_fwd_tc(pts, enc._flat_table(), geom, dirs, dir_group, mlp._flat_params(), dims, operand)
        ctx.enc, ctx.mlp, ctx.geom, ctx.dims, ctx.dir_group, ctx.operand = enc, mlp, geom, dims, dir_group, operand
        ctx.tab_grad = ParamGrad(enc, any(ctx.needs_input_grad[5:5 + enc.L]))
        ctx.mlp_grad = ParamGrad(mlp, any(ctx.needs_input_grad[5 + enc.L:]))
        ctx.save_for_backward(pts, dirs, feat16, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        pts, dirs, feat16, out = ctx.saved_tensors
        tab, mlp = ctx.tab_grad, ctx.mlp_grad
        g, dflat = tab.buffer(), mlp.buffer()
        ddirs = ops.field_bwd_tc(pts, ctx.geom, dirs, ctx.dir_group, ctx.mlp._flat_params(), ctx.dims, feat16, out.detach(),
                                 dout.float().contiguous(), g, ctx.needs_input_grad[1], dflat, operand=ctx.operand,
                                 grad_scale=ctx.mlp.tc_grad_scale)
        mlp.complete()
        tab.complete()
        return (None, ddirs, None, None, None) + tab.grads() + mlp.grads()


class _FieldRaysFn(torch.autograd.Function):
    """The autocast training path, one autograd node per field pass: (rays_o, rays_d, t) -> (R*S,4) [rgb, sigma].
    Forward: hbr_hash_encode_fwd_rays (sample positions formed in the kernel, features written once, already in the MLP's
    16-bit operand format -- the rounding MLP_3D's first Linear applies to its input under autocast, test_hash.py:53) ->
    hbr_mlp_fwd_tc.  Backward: hbr_mlp_bwd_tc (recomputes from the saved 16-bit features) -> hbr_hash_encode_bwd_rays.
    Against the module-by-module path (HashEncoder.forward -> MLP_3D.field) the (R*S,3) positions and the fp32 features are
    never written or read, and the MLP kernels skip their conversion pass; the arithmetic is the same."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, t, dirs, enc, mlp, *params):
        geom, dims = enc._geom(), mlp._dims()
        operand = ops.tc_operand()
        S = t.shape[-1]
        # the MLP's operand image is built on a side stream, beside the hash-grid kernel (in a captured step: a parallel
        # branch of the graph)
        cur, side = torch.cuda.current_stream(), _side_stream(rays_o.device)
        flat = mlp._flat_params()
        side.wait_stream(cur)
        if FUSE_GATHER and rays_o.shape[0] * S <= FUSE_GATHER_MAX_POINTS and ops.field_scatter_supported(geom, dims):
            # ONE kernel: the gather runs on dedicated warps of the MLP kernel and feeds its tile groups tile by tile
            # (hbr_field_fwd_rays_tc); it converts the parameters itself, so the operand image -- still wanted by the
            # backward -- is built beside it instead of in front of it
            out, feat16 = ops.field_fwd_rays_tc(rays_o, rays_d, t, enc._flat_table(), geom, dirs, flat, dims, operand)
            with torch.cuda.stream(side):
                ops.mlp_tc_prepare(flat, dims, operand)
            cur.wait_stream(side)
        else:
            with torch.cuda.stream(side):
                ops.mlp_tc_prepare(flat, dims, operand)
            feat16 = ops.hash_encode_fwd_rays(rays_o, rays_d, t, enc._flat_table(), geom, operand)
            cur.wait_stream(side)
            out, _ = ops.mlp_fwd_tc(feat16, dirs, S, flat, dims, operand=operand, image_ready=True)
        ctx.enc, ctx.mlp, ctx.geom, ctx.dims, ctx.S, ctx.operand = enc, mlp, geom, dims, S, operand
        ctx.save_for_backward(rays_o, rays_d, t, dirs, feat16, out)
        ctx.tab_grad = ParamGrad(enc, any(ctx.needs_input_grad[6:6 + enc.L]))
        ctx.mlp_grad = ParamGrad(mlp, any(ctx.needs_input_grad[6 + enc.L:]))
        return out

    @staticmethod
    def backward(ctx, dout):
        rays_o, rays_d, t, dirs, feat16, out = ctx.saved_tensors
        tab, mlp = ctx.tab_grad, ctx.mlp_grad
        flat = ctx.mlp._flat_params()
        dflat = mlp.buffer()
        n_pts = feat16.shape[0]
        # single GPU, the reference's configuration family: ONE kernel -- the scatter-add into the table gradient runs on
        # dedicated warps of the MLP backward kernel, tile by tile (hbr_field_bwd_rays_tc); the gradient exchange of the
        # multi-GPU path publishes level chunks of the table gradient while the scatter-add is still running, so it keeps
        # the two-kernel form below
        # (measured: 0.467 against 0.477 ms per 4 096-ray step; at 131 072 rays the two kernels, each at full occupancy,
        # are 1 % ahead, hence the size limit)
        if (FUSE_SCATTER and tab.wanted and mlp.wanted and tab.exchange is None and mlp.exchange is None
                and n_pts <= FUSE_SCATTER_MAX_POINTS and ops.field_scatter_supported(ctx.geom, ctx.dims)):
            g = tab.buffer()
            ddirs = ops.field_bwd_rays_tc(feat16, rays_o, rays_d, t, ctx.geom, dirs, flat, ctx.dims, out.detach(),
                                          dout.float().contiguous(), g, ctx.needs_input_grad[3], dflat, operand=ctx.operand,
                                          grad_scale=ctx.mlp.tc_grad_scale, defer_reduce=False)
            return (None, None, None, ddirs, None, None) + tab.grads() + mlp.grads()
        # the reduction of the MLP kernel's per-CTA gradient rows runs on a side stream, beside the hash-grid backward
        defer = tab.wanted
        # streamed exchange (dist.PeerGradAllReduce(streamed=True)): the last table backward of the pass finishes the table
        # gradient level chunk by level chunk while the all-reduce kernel beside it sends the finished chunks; the MLP kernel
        # then writes d(features) level-major for the level-major scatter-add
        plan = tab.stream_plan(n_pts)
        lm = plan is not None and STREAM_LEVEL_MAJOR and ops.mlp_level_major_ok(ctx.geom, ctx.dims, n_pts)
        dfeat, ddirs = ops.mlp_bwd_tc(feat16, dirs, ctx.S, flat, ctx.dims, out.detach(), dout.float().contiguous(), tab.wanted,
                                      ctx.needs_input_grad[3], dflat, operand=ctx.operand, grad_scale=ctx.mlp.tc_grad_scale,
                                      defer_reduce=defer, level_major=lm)
        cur, side = torch.cuda.current_stream(), _side_stream(dout.device)
        if defer:
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                ops.mlp_tc_reduce_grads(ctx.dims, n_pts, dflat, dout.device)
            dflat.record_stream(side)

        def join_mlp():
            if defer:
                cur.wait_stream(side)
            mlp.complete()

        def stream(g, chunks, done):
            if lm:
                ops.hash_encode_bwd_rays_lm(rays_o, rays_d, t, dfeat, ctx.geom, g, chunks, done)
                return ops.hash_bwd_lm_ctas(n_pts)
            ops.hash_encode_bwd_rays_stream(rays_o, rays_d, t, dfeat, ctx.geom, g, chunks, done)
            return ops.hash_bwd_stream_tiles(n_pts)

        if tab.wanted:
            # the MLP gradient is complete (and published) behind the first level chunk, or travels in the streamed exchange
            tab.scatter_table(lambda g, l0, l1: ops.hash_encode_bwd_rays(rays_o, rays_d, t, dfeat, ctx.geom, g, l0, l1),
                              n_pts, stream, after_first=join_mlp, mlp=mlp, mlp_stream=side if defer else None)
        else:
            join_mlp()
        return (None, None, None, ddirs, None, None) + tab.grads() + mlp.grads()


class _FieldCompactFn(torch.autograd.Function):
    """_FieldRaysFn with the occupancy grid as a live empty-space skipper (SURVEY 8f row 3): hbr_compact_samples keeps only
    the samples that fall into occupied cells; the encoder, the MLP and their backward passes run on that compacted list
    (live count on the device: no host synchronisation), and the compositor reads it back through the row map.  Skipped
    samples contribute exactly what the reference's masked path gives them (sigma = rgb = 0, vol_renderer.py:211-216)."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, t, dirs, grid, mu, sigma, enc, mlp, *params):
        geom, dims = enc._geom(), mlp._dims()
        operand = ops.tc_operand()
        pts_c, ray_c, rowmap, count = ops.compact_samples(rays_o, rays_d, t, grid, mu, sigma)
        cur, side = torch.cuda.current_stream(), _side_stream(rays_o.device)
        flat = mlp._flat_params()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            ops.mlp_tc_prepare(flat, dims, operand)
        feat16 = ops.hash_encode_fwd_pts(pts_c, count, enc._flat_table(), geom, operand)
        cur.wait_stream(side)
        out, _ = ops.mlp_fwd_tc(feat16, dirs, 1, flat, dims, operand=operand, image_ready=True, n_dev=count, dir_rows=ray_c)
        ctx.enc, ctx.mlp, ctx.geom, ctx.dims, ctx.operand = enc, mlp, geom, dims, operand
        ctx.save_for_backward(pts_c, ray_c, count, dirs, feat16, out)
        ctx.tab_grad = ParamGrad(enc, any(ctx.needs_input_grad[9:9 + enc.L]))
        ctx.mlp_grad = ParamGrad(mlp, any(ctx.needs_input_grad[9 + enc.L:]))
        ctx.mark_non_differentiable(rowmap, count)
        return out, rowmap, count

    @staticmethod
    def backward(ctx, dout, _g_rowmap, _g_count):
        pts_c, ray_c, count, dirs, feat16, out = ctx.saved_tensors
        tab, mlp = ctx.tab_grad, ctx.mlp_grad
        dflat = mlp.buffer()
        dfeat, ddirs = ops.mlp_bwd_tc(feat16, dirs, 1, ctx.mlp._flat_params(), ctx.dims, out.detach(), dout.float().contiguous(),
                                      tab.wanted, ctx.needs_input_grad[3], dflat, operand=ctx.operand,
                                      grad_scale=ctx.mlp.tc_grad_scale, n_dev=count, dir_rows=ray_c)
        mlp.complete()
        if tab.wanted:
            ops.hash_encode_bwd_pts(pts_c, count, dfeat, ctx.geom, tab.buffer(), 0, ctx.enc.L)
            tab.complete()                                 # published whole
        return (None, None, None, ddirs, None, None, None, None, None) + tab.grads() + mlp.grads()


# hbr_field_bwd_rays_tc (MLP backward + hash-grid scatter-add in one kernel) on the single-GPU autocast path; the
# environment switch exists for A/B measurements (bench.py --no-fuse-scatter)
FUSE_SCATTER = os.environ.get("HBR_FUSE_SCATTER", "1") != "0"
FUSE_SCATTER_MAX_POINTS = 1 << 21
# hbr_field_fwd_rays_tc (hash-grid gather + MLP forward in one kernel) on the autocast path: opt-in.  Measured at 4 096 rays x
# 128 samples: 152 us with 8 gather warps beside two tile groups, 162 us with 16 (setmaxnreg 128 / 56), against 108 + 32 us
# for the two kernels -- bit-identical results; the layer chain of only two tile groups, sharing the issue slots with the
# gather's address arithmetic, becomes the bottleneck (bench.py --fuse-gather)
FUSE_GATHER = os.environ.get("HBR_FUSE_GATHER", "0") != "0"
FUSE_GATHER_MAX_POINTS = 1 << 21
# streamed gradient exchange (multi-GPU): producer = the level-major scatter-add (co-resident grid walking the levels in
# order, hbr_hash_encode_bwd_rays_lm) or the tile-major kernel launched chunk-major (hbr_hash_encode_bwd_rays_stream)
# (measured on 8 GPUs, 4 096 rays each: tile-major in 4 equal level chunks 0.594 ms per step, level-major in 8 chunks 0.685 --
# its 512 persistent CTAs fill the register file and keep the exchange kernel waiting --, one launch pair per chunk 0.639)
STREAM_LEVEL_MAJOR = os.environ.get("HBR_STREAM_LEVEL_MAJOR", "0") != "0"

_SIDE = {}


def _side_stream(device) -> torch.cuda.Stream:
    """One side stream per device for the small kernels that can run beside the hash-grid kernels."""
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    s = _SIDE.get(idx)
    if s is None:
        s = _SIDE[idx] = torch.cuda.Stream(device=idx)
    return s


# Volume_Renderer.render: colours, depth and opacity maps of the coarse and the fine pass, the eikonal norms (SDF mode)
RenderOut = namedtuple("RenderOut", "rgb_coarse rgb_fine depth_coarse depth_fine opacity_coarse opacity_fine norm")


def _unwrap(model):
    if isinstance(model, nn.DataParallel) and len(model.device_ids) <= 1:
        return model.module
    return model


class Volume_Renderer:
    def __init__(self, H, W, K, near=0., far=1., device=None, Pos_encode=None, Dir_encode=None, max_dim=1024,
                 sigma_val=torch.as_tensor(1), mu=torch.as_tensor(0), use_sdf: Optional[bool] = False,
                 var_model: Optional[nn.Module] = None):
        self.H, self.W, self.K = H, W, K
        self.near, self.far = near, far
        self.device = device
        if device is None:
            self.device = "cuda" if torch.cuda.is_available() else "cpu"
        self.coods_x, self.coords_y = torch.meshgrid(torch.arange(W, device=self.device), torch.arange(H, device=self.device),
                                                     indexing="xy")
        self.Pos_encode = Pos_encode
        self.Dir_encode = Dir_encode
        self.grid_size = max_dim // 4
        g = self.grid_size
        self.bool_grid = torch.ones((g, g, g), device=self.device, dtype=torch.bool)      # vol_renderer.py:107
        self.sigma_val = sigma_val.to(self.device)
        self.mu = mu.to(self.device)
        self.epislon = 1e-5
        self.tmp_arr = torch.zeros((g, g, g), device=self.device, dtype=torch.int8)
        self.reset_mask = False
        self.use_sdf = use_sdf
        self.var_model = var_model
        self._dp_checked = False
        self._grid_flags = None
        # vol_render feeds the kernels at most this many sample points at a time (ray chunks): per-point temporaries of a
        # 2^20-ray step would otherwise be tens of GB (SURVEY H10).  2^26 points = 524 288 rays x 128 samples.
        self.max_points = 1 << 26
        # SURVEY 8f row 3: with an occupancy grid that is not all-True, True = skip the samples outside occupied cells
        # altogether (compacted sample lists through encoder, MLP and compositor) instead of evaluating and zeroing them;
        # same numbers, work proportional to the live samples.  Autocast / native modules only; off by default.
        self.compact = False
        self._grid_state = (None, True)           # (bool_grid._version, all_true)
        self._host_norm = None
        # Encoder + MLP fused into one kernel per direction (hbr_field_*_tc): no fp32 feature / d(feature) tensors in HBM
        # (-235 B/point of traffic), same results.  Measured on B200 at 4096 x 128 points it is time-neutral against the
        # separate kernels (the tile groups of the tensor-core kernel run at low occupancy, so their gather / scatter
        # phases are latency-bound), and the separate path can overlap the table-gradient all-reduce per level chunk,
        # so it is opt-in: True fuses whenever the configuration is covered, "auto" only without gradient hooks.
        self.fuse_field = False
        # Under autocast one autograd node drives the separate kernels (_FieldRaysFn): sample positions formed inside the
        # hash-grid kernels, features handed to the MLP kernels in their 16-bit operand format.  False = module by module
        # (HashEncoder.forward -> MLP_3D.field), the path every other caller of those modules takes.
        self.chain_field = True
        # Early ray termination in the compositor (north star kernel 3; SURVEY H8): opt-in.  True skips the 32-sample chunks
        # behind the point where the accumulated optical depth exceeds ops.ERT_TAU = 104, i.e. where the transmittance is
        # exactly 0 in fp32; identical results whenever the depth does not fall back below it (always for sigma >= 0 -- the
        # reference's LeakyReLU density can be slightly negative, hence off by default).
        self.ert = False
        # SDF mode (use_sdf) with the native modules and the reference's VarModel: the field runs as in NeRF mode and the
        # SDF compositing / eikonal stencil kernels of csrc/sdf.cu take its packed output (False: the reference's data flow,
        # _generic, whose calc_color still uses those kernels).  hierarchical=True stays on _generic: it fails there exactly
        # like the reference does (vol_renderer.py:242 passes no sample positions).
        self.sdf_native = True

    # -- occupancy grid (vol_renderer.py:116-140) --------------------------------------------------------------
    def update_grid(self, points: torch.Tensor, alpha: torch.Tensor):
        """vol_renderer.py:116-131.  CUDA tensors go through hbr_occupancy_update (one pass, the "nothing was hit -> whole
        grid True" fallback decided on the device, no synchronisation); the alpha <= 0 -> 0 clamp is applied to the
        caller's tensor like the reference does."""
        if points.is_cuda and self.bool_grid.is_cuda and self.mu.numel() in (1, 3):
            alpha[alpha <= 0] = 0                                             # :121, in place on the caller's tensor
            mu, sig = self._norm_host()
            if self._grid_flags is None or self._grid_flags.device != self.bool_grid.device:
                self._grid_flags = torch.zeros(2, dtype=torch.int32, device=self.bool_grid.device)
            ops.occupancy_update(points, alpha, self.bool_grid, mu, sig, self._grid_flags)
            self._grid_state = (None, True)                                   # contents changed behind torch's version counter
            return
        points = (points - self.mu) / self.sigma_val
        points = (points * self.grid_size).long()
        alpha[alpha <= 0] = 0
        self.tmp_arr[points[..., 0], points[..., 1], points[..., 2]] += torch.ceil(alpha).int()
        if torch.sum(self.tmp_arr > 0) == 0:
            self.bool_grid[...] = True
        else:
            self.bool_grid[self.tmp_arr > 0] = True
        self.tmp_arr[self.tmp_arr > 0] = 0

    def _norm_host(self):
        if self._host_norm is None:
            mu = self.mu.detach().reshape(-1).float().cpu().tolist()
            if len(mu) == 1:
                mu = mu * 3
            self._host_norm = (mu, float(self.sigma_val.detach().cpu()))
        return self._host_norm

    @torch.no_grad()
    def update_grid_from_field(self, model, threshold: float = 0.01, chunk: int = 1 << 21, reset: bool = True):
        """Make the occupancy grid LIVE: evaluate the density of the current field at the centre of every grid cell
        (cell (i,j,k) covers ((p - mu) / sigma * G) in [i, i+1) x ..., the arithmetic of get_mask) and mark the cells whose
        density exceeds `threshold` (reset=True clears the grid first, like reset_mask at vol_renderer.py:201-203).  With
        `self.compact = True` the training step then skips every sample outside the marked cells.  The reference never
        refreshes its grid (update_grid is commented out of vol_render, :205) -- this is SURVEY 8f row 3."""
        mlp = self._native(model)
        if mlp is None:
            raise TypeError("update_grid_from_field needs the native HashEncoder / MLP_3D")
        G = self.grid_size
        dev = self.bool_grid.device
        mu, sig = self._norm_host()
        if reset:
            self.bool_grid[...] = False
        idx = torch.arange(G, device=dev, dtype=torch.float32) + 0.5
        mu_t = torch.tensor(mu, device=dev)
        flat = self.bool_grid.view(-1)
        for i0 in range(0, G, max(1, chunk // (G * G))):
            i1 = min(G, i0 + max(1, chunk // (G * G)))
            ii, jj, kk = torch.meshgrid(idx[i0:i1], idx, idx, indexing="ij")
            p = torch.stack((ii, jj, kk), dim=-1).reshape(-1, 3) / G * sig + mu_t
            dens = mlp(self.Pos_encode(p))                                       # density-only branch, fp32 kernels
            flat[i0 * G * G:i1 * G * G] |= dens.reshape(-1) > threshold
        self._grid_state = (None, True)
        return float(self.bool_grid.float().mean())

    def get_mask(self, points: torch.Tensor) -> torch.Tensor:
        mu, sig = self._norm_host()
        return ops.occupancy_mask(points, self.bool_grid, mu, sig)

    def _grid_all_true(self) -> bool:
        ver = self.bool_grid._version
        if self._grid_state[0] != (ver, self.bool_grid.data_ptr()):
            self._grid_state = ((ver, self.bool_grid.data_ptr()), bool(self.bool_grid.all()))   # one sync per grid edit
        return self._grid_state[1]

    # -- the hot path ----------------------------------------------------------------------------------------
    def _native(self, model):
        m = _unwrap(model)
        ok = (isinstance(self.Pos_encode, HashEncoder) and isinstance(self.Dir_encode, PositionalEncoder)
              and isinstance(m, MLP_3D) and m._native and not m.use_sdf and not self.use_sdf)
        return m if ok else None

    def _can_fuse(self, mlp) -> bool:
        enc = self.Pos_encode
        if self.fuse_field is False or not (torch.is_autocast_enabled() and ops.HAS_TC):
            return False
        ok = (enc.F == 2 and enc.L == 16 and enc.E == 0 and enc.T >= 2 and (enc.T & (enc.T - 1)) == 0
              and mlp._in0 == 32 and mlp.d_view <= 25)
        if self.fuse_field == "auto":
            ok = ok and enc._dp is None
        return ok

    def _ert_tau(self) -> float:
        return ops.ERT_TAU if self.ert else 0.0

    def _can_chain(self, mlp) -> bool:
        """_FieldRaysFn covers the autocast path whenever the encoder's width is the MLP kernels' operand width."""
        enc = self.Pos_encode
        if not (self.chain_field and torch.is_autocast_enabled() and ops.HAS_TC):
            return False
        width = enc.L * enc.F + enc.E
        return width == mlp._in0 and (width % 2 == 0) and ((width == 32 and mlp.d_view <= 25) or width == 64)

    def _composite(self, out4, t, dir_norm, mask, R, S, rowmap=None, maps=False):
        if maps:
            return ops.CompositeMapsPacked.apply(out4, t, dir_norm, mask, R, S, self._ert_tau(), rowmap)
        return ops.CompositePacked.apply(out4, t, dir_norm, mask, R, S, self._ert_tau(), rowmap)

    def _field_pass(self, mlp, rays_o, rays_d, t, dir_enc, dir_norm, mask_needed, maps=False):
        """positions -> encoder -> MLP -> compositing for depths t ((S,) shared or (R,S) per ray) -> (C, w), or with maps
        (C, w, depth, opacity)."""
        R, S = rays_o.shape[0], t.shape[-1]
        if not self._can_fuse(mlp) and self._can_chain(mlp):
            enc = self.Pos_encode
            if enc._flat_table().device != rays_o.device:
                raise RuntimeError(f"encoder tables are on {enc._flat_table().device}, rays on {rays_o.device}")
            if mask_needed and self.compact and S <= 1024 and R * S < 2 ** 31:
                mu, sig = self._norm_host()
                out4, rowmap, _ = _FieldCompactFn.apply(rays_o, rays_d, t.float().contiguous(), dir_enc.float().contiguous(),
                                                        self.bool_grid, mu, sig, enc, mlp, *node_params(enc, mlp))
                return self._composite(out4, t, dir_norm, None, R, S, rowmap, maps)
            mask = self.get_mask(ops.ray_points(rays_o, rays_d, t).view(-1, 3)) if mask_needed else None
            out4 = _FieldRaysFn.apply(rays_o, rays_d, t.float().contiguous(), dir_enc.float().contiguous(), enc, mlp,
                                      *node_params(enc, mlp))
            return self._composite(out4, t, dir_norm, mask, R, S, None, maps)
        pts = ops.ray_points(rays_o, rays_d, t).view(-1, 3)
        mask = self.get_mask(pts) if mask_needed else None
        if self._can_fuse(mlp):
            enc = self.Pos_encode
            if enc._flat_table().device != pts.device:
                raise RuntimeError(f"encoder tables are on {enc._flat_table().device}, rays on {pts.device}")
            out4 = _FieldFn.apply(pts, dir_enc, S, enc, mlp, *node_params(enc, mlp))
        else:
            feat = self.Pos_encode(pts)
            out4 = mlp.field(feat, dir_enc, S)
        return self._composite(out4, t, dir_norm, mask, R, S, None, maps)

    def vol_render(self, model, rays_d: torch.Tensor, rays_o: torch.Tensor, num_samples=100,
                   t: Optional[torch.Tensor] = None, update_mask=False, dir_norm=1, hierarchical=True,
                   _u=None, _u_cand=None) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
        if not rays_d.is_cuda:
            raise RuntimeError("Volume_Renderer.vol_render needs CUDA tensors (there is no CPU fallback)")
        near, far = self.near, self.far
        device = "cuda"
        if t is None:
            t = strat_sampler(near, far, num_samples, device=rays_d.device)                 # RNG draw #1
        if self.use_sdf and self.sdf_native and hierarchical is not True and update_mask is not True and t.shape[-1] <= 1024:
            sdf_mlp = self._native_sdf(model)
            if sdf_mlp is not None and self._grid_all_true():
                self._auto_dp(sdf_mlp)
                return self._render_sdf(sdf_mlp, rays_o, rays_d, t)
        mlp = self._native(model)
        if mlp is not None:
            self._auto_dp(mlp)
        if mlp is None:
            return self._generic(model, rays_d, rays_o, t, update_mask, dir_norm, hierarchical, _u, _u_cand)

        rays_o = rays_o.float().contiguous()
        rays_d = rays_d.float().contiguous()
        dir_enc = self.Dir_encode(rays_d)                                                      # (R, 2*3*num_freq), once per ray
        if update_mask is True:
            if self.reset_mask is True:                                                        # vol_renderer.py:201-203
                self.bool_grid[...] = False
                self.reset_mask = False
            mask_needed = False
        else:
            mask_needed = not self._grid_all_true()
        R, S = rays_o.shape[0], t.shape[-1]
        per = max(1, int(self.max_points) // (S * (3 if hierarchical is True else 1)))
        if R > per:
            # Large batches (BASELINE configs[2]: 2^20 rays/step) go through the kernels in ray chunks (SURVEY H10): the
            # per-point temporaries (features, d(features), field outputs) exist for one chunk at a time.  The RNG draws of
            # the hierarchical resampler are made ONCE for the whole batch, in the reference's order, and sliced.
            if hierarchical is True and _u is None:
                _u = torch.rand((R, S), device=rays_o.device)                                  # RNG draw #2 (helper.py:40)
                _u_cand = torch.rand(S, device=rays_o.device)                                  # RNG draw #3 (helper.py:43)
            dn_rows = torch.is_tensor(dir_norm) and dir_norm.numel() == R
            Crs, Cfs = [], []
            for r0 in range(0, R, per):
                sl = slice(r0, min(R, r0 + per))
                cr, cf = self._render_rays(mlp, rays_o[sl], rays_d[sl], t, dir_enc[sl], dir_norm[sl] if dn_rows else dir_norm,
                                           mask_needed, hierarchical, _u[sl] if _u is not None else None, _u_cand)
                Crs.append(cr)
                Cfs.append(cf)
            Cr = torch.cat(Crs)
            return Cr, (Cr if hierarchical is not True else torch.cat(Cfs)), None
        Cr, Cf = self._render_rays(mlp, rays_o, rays_d, t, dir_enc, dir_norm, mask_needed, hierarchical, _u, _u_cand)
        return Cr, Cf, None

    def render(self, model, rays_d: torch.Tensor, rays_o: torch.Tensor, num_samples=100, t: Optional[torch.Tensor] = None,
               dir_norm=1, hierarchical=True) -> RenderOut:
        """vol_render with depth and opacity maps: RenderOut(rgb_coarse, rgb_fine, depth_coarse, depth_fine, opacity_coarse,
        opacity_fine, norm).  Same RNG draws, routes (chained, fused, compact, masked, early ray termination) and ray chunks
        as vol_render(update_mask=False), so the colours are bit-identical to vol_render's; without hierarchical the fine
        outputs are the coarse ones.
          depth = sum_s w_s t_s: distance along the unit ray direction, in the units of t (p = o + d t, |d| = 1 as get_od
                  and ops.ray_gen return it).  z-depth along the camera axis is depth / dir_norm.
          opacity = sum_s w_s: what a person-mask loss supervises.
        Neither is normalised by the opacity or clamped: MLP_3D's LeakyReLU density can be slightly negative, so weights and
        opacity can leave [0, 1].  Both carry gradients (to the tables and the MLP through the compositor's backward).
        Native modules only: the NeRF route (HashEncoder / PositionalEncoder / MLP_3D) and the native SDF route
        (hierarchical=False, reference VarModel; norm = eikonal norms, maps from the SDF weights); anything else raises
        TypeError."""
        if not rays_d.is_cuda:
            raise RuntimeError("Volume_Renderer.render needs CUDA tensors (there is no CPU fallback)")
        if t is None:
            t = strat_sampler(self.near, self.far, num_samples, device=rays_d.device)                 # RNG draw #1
        if self.use_sdf:
            sdf_mlp = self._native_sdf(model) if (self.sdf_native and hierarchical is not True and t.shape[-1] <= 1024) else None
            if sdf_mlp is None or not self._grid_all_true():
                raise TypeError("Volume_Renderer.render in SDF mode needs the native SDF route: HashEncoder / "
                                "PositionalEncoder / MLP_3D with the reference's VarModel, hierarchical=False, at most 1024 "
                                "samples and an all-True occupancy grid")
            self._auto_dp(sdf_mlp)
            Cr, w, norm = self._sdf_pass(sdf_mlp, rays_o, rays_d, t)
            D, A = (w * t).sum(-1), w.sum(-1)
            return RenderOut(Cr, Cr, D, D, A, A, norm)
        mlp = self._native(model)
        if mlp is None:
            raise TypeError("Volume_Renderer.render needs the native HashEncoder / PositionalEncoder / MLP_3D")
        self._auto_dp(mlp)
        rays_o = rays_o.float().contiguous()
        rays_d = rays_d.float().contiguous()
        dir_enc = self.Dir_encode(rays_d)
        mask_needed = not self._grid_all_true()
        R, S = rays_o.shape[0], t.shape[-1]
        per = max(1, int(self.max_points) // (S * (3 if hierarchical is True else 1)))
        if R > per:
            _u = _u_cand = None
            if hierarchical is True:                                        # drawn once for the batch, as vol_render does
                _u = torch.rand((R, S), device=rays_o.device)                                  # RNG draw #2
                _u_cand = torch.rand(S, device=rays_o.device)                                  # RNG draw #3
            dn_rows = torch.is_tensor(dir_norm) and dir_norm.numel() == R
            parts = []
            for r0 in range(0, R, per):
                sl = slice(r0, min(R, r0 + per))
                parts.append(self._render_rays(mlp, rays_o[sl], rays_d[sl], t, dir_enc[sl], dir_norm[sl] if dn_rows else dir_norm,
                                               mask_needed, hierarchical, _u[sl] if _u is not None else None, _u_cand, maps=True))
            out = [torch.cat(c) for c in zip(*parts)]
            return RenderOut(*out, None)
        return RenderOut(*self._render_rays(mlp, rays_o, rays_d, t, dir_enc, dir_norm, mask_needed, hierarchical, None, None,
                                            maps=True), None)

    @torch.no_grad()
    def render_view(self, model, c2w, num_samples, hierarchical=True, chunk=1 << 16, t: Optional[torch.Tensor] = None):
        """Whole views from camera poses: c2w (4,4) or (V,4,4), the renderer's H, W, K.  Rays are generated on the device
        (ops.ray_gen) chunk by chunk -- `chunk` rays at a time, never V*H*W at once -- and each chunk is one render() call
        (dir_norm = the ray generator's direction norm).  Returns rgb (V,H,W,3) (the fine colour when hierarchical), depth
        (V,H,W) and opacity (V,H,W), from the fine pass when hierarchical.  Runs under no_grad; without `t` every chunk
        draws its own stratified depths, so the result depends on `chunk` exactly as the RNG stream does."""
        dev = self.bool_grid.device
        if dev.type != "cuda":
            raise RuntimeError("Volume_Renderer.render_view needs a CUDA device (there is no CPU fallback)")
        c2w = torch.as_tensor(c2w).to(dev, torch.float32)
        if c2w.dim() == 2:
            c2w = c2w[None]
        if c2w.shape[1:] != (4, 4):
            raise ValueError("c2w must be (4,4) or (V,4,4)")
        V, H, W = c2w.shape[0], int(self.H), int(self.W)
        n = V * H * W
        chunk = max(1, int(chunk))
        rgb = torch.empty((n, 3), device=dev, dtype=torch.float32)
        depth = torch.empty((n,), device=dev, dtype=torch.float32)
        opacity = torch.empty((n,), device=dev, dtype=torch.float32)
        for first in range(0, n, chunk):
            m = min(chunk, n - first)
            o, d, nrm, _ = ops.ray_gen(c2w, H, W, self.K, first=first, n_rays=m)
            out = self.render(model, d, o, num_samples, t=t, dir_norm=nrm, hierarchical=hierarchical)
            rgb[first:first + m] = out.rgb_fine
            depth[first:first + m] = out.depth_fine
            opacity[first:first + m] = out.opacity_fine
        return rgb.view(V, H, W, 3), depth.view(V, H, W), opacity.view(V, H, W)

    def _auto_dp(self, mlp):
        """launch_rank.py's zero-edit multi-GPU run of the trainer (HBR_AUTO_DP=1): at the first native render of a process
        that belongs to a process group, take rank 0's parameters and attach the gradient exchange (dist.auto_attach);
        SDF mode's VarModel parameter joins through a small all-reduce of its own."""
        if self._dp_checked:
            return
        self._dp_checked = True
        if os.environ.get("HBR_AUTO_DP") == "1":
            from . import dist as _hdist
            extra = list(self.var_model.parameters()) if (self.use_sdf and isinstance(self.var_model, nn.Module)) else ()
            _hdist.auto_attach(self.Pos_encode, mlp, extra=extra)

    # -- SDF mode on the native modules (SURVEY 8f row 4; vol_renderer.py:165-223 with use_sdf -> helper.py:76-89) -----
    def _native_sdf(self, model):
        from .helper import VarModel
        m = _unwrap(model)
        ok = (isinstance(self.Pos_encode, HashEncoder) and isinstance(self.Dir_encode, PositionalEncoder)
              and isinstance(m, MLP_3D) and m._native and type(self.var_model) is VarModel)
        return m if ok else None

    def _render_sdf(self, mlp, rays_o, rays_d, t):
        """One coarse pass in SDF mode: the field as in NeRF mode (directions encoded once per ray, packed (N,4) output with
        the density head's LeakyReLU value in column 3), then hbr_composite_sdf_* forms 2*sigmoid - 1 and composites in one
        kernel each way, and the eikonal norms come from the 6-point stencil (MLP_3D.eikonal_norms).  dir_norm plays no
        part (helper.py:71 computes del_t, the SDF branch never reads it).  Returns (Cr, Cr, norm) like the reference."""
        Cr, _, norm = self._sdf_pass(mlp, rays_o, rays_d, t)
        return Cr, Cr, norm

    def _sdf_pass(self, mlp, rays_o, rays_d, t):
        """_render_sdf's pass -> (Cr, w (R,S) with a gradient, eikonal norms)."""
        rays_o = rays_o.float().contiguous()
        rays_d = rays_d.float().contiguous()
        dir_enc = self.Dir_encode(rays_d)
        R, S = rays_o.shape[0], t.shape[-1]
        enc = self.Pos_encode
        pts = ops.ray_points(rays_o, rays_d, t).view(-1, 3)
        if self._can_chain(mlp):
            out4 = _FieldRaysFn.apply(rays_o, rays_d, t.float().contiguous(), dir_enc.float().contiguous(), enc, mlp,
                                      *node_params(enc, mlp))
        else:
            out4 = mlp.field(enc(pts), dir_enc, S, raw=True)
        Cr, w = ops.CompositeSdfPacked.apply(out4, self.var_model.b, R, S, bool(mlp.use_sdf))
        norm = mlp.eikonal_norms(pts, encoder=enc)
        return Cr, w, norm

    def _render_rays(self, mlp, rays_o, rays_d, t, dir_enc, dir_norm, mask_needed, hierarchical, _u, _u_cand, maps=False):
        """-> (Cr, Cf), or with maps (Cr, Cf, depth_r, depth_f, opacity_r, opacity_f)."""
        coarse = self._field_pass(mlp, rays_o, rays_d, t, dir_enc, dir_norm, mask_needed, maps)
        Cr, w = coarse[0], coarse[1]
        if hierarchical is True:
            _, t_fine = hierarchical_sampling(rays_o, rays_d, z_vals=t, weights=w, n_samples=t.shape[-1], tn=self.near,
                                              tf=self.far, device="cuda", _u=_u, _u_cand=_u_cand)   # RNG draws #2, #3
            fine = self._field_pass(mlp, rays_o, rays_d, t_fine, dir_enc, dir_norm, False, maps)  # the fine pass never masks (:237)
        else:
            fine = coarse
        if maps:
            return Cr, fine[0], coarse[2], fine[2], coarse[3], fine[3]
        return Cr, fine[0]

    def _generic(self, model, rays_d, rays_o, t, update_mask, dir_norm, hierarchical, _u, _u_cand):
        """Reference data flow for foreign encoders / models (vol_renderer.py:165-245)."""
        Pos_encode, Dir_encode = self.Pos_encode, self.Dir_encode
        if Pos_encode is None:
            raise ValueError("ERROR: No positional encoding")                               # :191-192
        num_samples = t.shape[-1]

        def run(tt, masked, with_rays=True):
            pts = ops.ray_points(rays_o, rays_d, tt)
            R, S = pts.shape[0], pts.shape[1]
            flat = pts.reshape(-1, 3)
            dirs = rays_d[..., None, :].repeat(1, S, 1).reshape(-1, 3)
            enc = Pos_encode(flat)
            enc = enc.reshape(enc.shape[0], -1)
            if Dir_encode is not None:
                dirs = Dir_encode(dirs)
                dirs = dirs.reshape(dirs.shape[0], -1)
            if masked:
                mask = self.get_mask(flat)
                mo = model(enc[mask], dirs[mask])
                sigma = torch.zeros((R * S, 1), device=flat.device, dtype=mo.dtype)
                rgb = torch.zeros((R * S, 3), device=flat.device, dtype=mo.dtype)
                sigma[mask] = mo[..., 3:4]
                rgb[mask] = mo[..., 0:3]
            else:
                mo = model(enc, dirs)
                sigma, rgb = mo[..., 3:4], mo[..., 0:3]
            return calc_color(t=tt, rgb=rgb.reshape(R, S, -1), sigma=sigma.reshape(R, S), dir_norm=dir_norm,
                              use_sdf=self.use_sdf, var_model=self.var_model, rays=flat if with_rays else None, model=model,
                              encoder=Pos_encode)

        if update_mask is True and self.reset_mask is True:
            self.bool_grid[...] = False
            self.reset_mask = False
        Cr, wts, norm = run(t, update_mask is not True)
        if hierarchical is True:
            _, t_fine = hierarchical_sampling(rays_o, rays_d, z_vals=t, weights=wts, n_samples=num_samples, tn=self.near,
                                              tf=self.far, _u=_u, _u_cand=_u_cand)
            Cf, _, norm = run(t_fine, False, with_rays=False)          # vol_renderer.py:242 passes no sample positions
        else:
            Cf = Cr
        return Cr, Cf, norm


def make_batch(in_rays: torch.Tensor, batch_size: int) -> list:
    """vol_renderer.py:249-256."""
    return [in_rays[i:i + batch_size].to("cpu") for i in range(0, in_rays.shape[0], batch_size)]
