"""Drop-in for the model half of the reference's test_hash.py: `MLP_3D` (test_hash.py:20-105).

Same constructor, `forward(x, viewdirs=None, mask=None)`, state_dict keys (`sig_model.{0,2,4}.*`,
`col_model.{0,2,4}.*`) and RNG consumption at construction.  The twelve parameter tensors are views into
one flat fp32 buffer (state_dict order) that the kernels read directly.

Precision: fp32 CUDA-core kernels by default (nerf2mesh.py runs the field without autocast); under
`torch.autocast` the forward/backward run on the tcgen05 tensor-core kernels with bf16 operands and fp32
accumulation (the reference runs fp16 there, train_hash2.py:218).

Only the shape the reference instantiates -- num_sig=2, num_col=2, h_size=64 (train_hash2.py:127,
nerf2mesh.py:57) -- has a native implementation; anything else raises NotImplementedError.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from ._lib import MlpDims
from .dist import ParamGrad, node_params


class _MlpFn(torch.autograd.Function):
    """feat (N,in0), dirs (N/dir_group, d_view) -> (N,4) [rgb, sigma]."""

    @staticmethod
    def forward(ctx, feat, dirs, dir_group, mlp, use_tc, *params):
        flat = mlp._flat_params()
        dims = mlp._dims()
        train = any(ctx.needs_input_grad)
        feat = feat.float().contiguous()
        dirs = dirs.float().contiguous()
        if use_tc:
            out, act = ops.mlp_fwd_tc(feat, dirs, dir_group, flat, dims, keep_act=train, operand=use_tc)
        else:
            out, act = ops.mlp_fwd_f32(feat, dirs, dir_group, flat, dims, keep_act=train)
        ctx.grad = ParamGrad(mlp, any(ctx.needs_input_grad[5:]))
        ctx.mlp, ctx.dims, ctx.dir_group, ctx.use_tc = mlp, dims, dir_group, use_tc
        ctx.save_for_backward(feat, dirs, out if use_tc else act)     # the tensor-core backward reads the saved output
        return out

    @staticmethod
    def backward(ctx, dout):
        feat, dirs, act = ctx.saved_tensors
        mlp = ctx.mlp
        flat = mlp._flat_params()
        dflat = ctx.grad.buffer()
        dout = dout.float().contiguous()
        want_dfeat, want_ddirs = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if ctx.use_tc:
            dfeat, ddirs = ops.mlp_bwd_tc(feat, dirs, ctx.dir_group, flat, ctx.dims, act.detach(), dout, want_dfeat, want_ddirs,
                                          dflat, operand=ctx.use_tc, grad_scale=mlp.tc_grad_scale)
        else:
            dfeat, ddirs = ops.mlp_bwd_f32(feat, dirs, ctx.dir_group, flat, ctx.dims, dout, act, want_dfeat, want_ddirs, dflat)
        ctx.grad.complete()
        return (dfeat, ddirs, None, None, None) + ctx.grad.grads()


class _DensityFn(torch.autograd.Function):
    """feat (N,in0) -> (N,1) LeakyReLU density, the density-only branch (test_hash.py:73-77) WITH a backward: fp32 kernels,
    only the density head is evaluated and differentiated (hbr_mlp_fwd_f32 / hbr_mlp_bwd_f32 with dirs == NULL).  Serves
    SDF mode's eikonal stencil, where six of these per sample are the bulk of the step."""

    @staticmethod
    def forward(ctx, feat, mlp, *params):
        flat = mlp._flat_params()
        dims = mlp._dims()
        train = any(ctx.needs_input_grad)
        feat = feat.float().contiguous()
        out, act = ops.mlp_fwd_f32(feat, None, 1, flat, dims, keep_act=train)
        ctx.grad = ParamGrad(mlp, any(ctx.needs_input_grad[2:]))
        ctx.mlp, ctx.dims = mlp, dims
        ctx.save_for_backward(feat, act)
        return out

    @staticmethod
    def backward(ctx, dout):
        feat, act = ctx.saved_tensors
        flat = ctx.mlp._flat_params()
        dflat = ctx.grad.buffer()
        dfeat, _ = ops.mlp_bwd_f32(feat, None, 1, flat, ctx.dims, dout.float().contiguous(), act, ctx.needs_input_grad[0], False,
                                   dflat)
        ctx.grad.complete()
        return (dfeat, None) + ctx.grad.grads()


class MLP_3D(nn.Module):
    def __init__(self, num_sig=3, num_col=2, h_size=64, d_view=3, L=16, F=2, E=0, use_sdf=False, max_bound=1.0,
                 min_bound=-1.0):
        super().__init__()
        self.d_view = d_view
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        self.max_bound = torch.as_tensor(max_bound).to(dev)          # test_hash.py:25-26
        self.min_bound = torch.as_tensor(min_bound).to(dev)
        sig = [nn.Linear(L * F + E, h_size), nn.ReLU()]
        for i in range(num_sig):
            if i == num_sig - 1:
                sig.append(nn.Linear(h_size, 1 + 15))
            else:
                sig += [nn.Linear(h_size, h_size), nn.ReLU()]
        self.sigmoid = nn.Sigmoid()
        self.sig_model = nn.Sequential(*sig)
        self.relu, self.elu, self.lrelu = nn.ReLU(), nn.ELU(), nn.LeakyReLU()
        col = [nn.Linear(15 + d_view, h_size), nn.ReLU()]
        for i in range(num_col):
            if i == num_col - 1:
                col.append(nn.Linear(h_size, 3))
            else:
                col += [nn.Linear(h_size, h_size), nn.ReLU()]
        self.col_model = nn.Sequential(*col)
        self.use_sdf = use_sdf
        self._native = (num_sig == 2 and num_col == 2 and h_size == 64 and L * F + E <= 64 and 15 + d_view <= 64)
        self._in0 = L * F + E
        # power-of-two factor the tensor-core backward applies to the upstream gradient before rounding it to the 16-bit
        # operand format (and divides out of its results).  The reference's trainer scales the loss with GradScaler
        # (train_hash2.py:156,226), which does the same job from outside; set this when running fp16 operands without one.
        self.tc_grad_scale = 1.0
        # SDF mode: forward_sdf / the eikonal stencil always run the fp32 kernels (central differences with eps = 5e-4
        # amplify the density head's rounding 1000x).  The reference evaluates them inside torch.autocast like everything
        # else (train_hash2.py:218 -> helper.py:87), i.e. with fp16 matrix products; True follows it: under autocast the
        # training-time stencil pass runs on the 16-bit tensor-core kernels (measured 4096 x 128 samples x 6 stencil points:
        # profiles/r02f_sdf_measurements.json).  Off by default.
        self.sdf_follows_autocast = False
        self._dp = None               # the data-parallel gradient exchange attached to this module (dist._GradExchange)
        self._flat = None
        if self._native:
            self._reflatten()

    # -- flat parameter storage ----------------------------------------------------------------------------
    def _ordered(self):
        ps = []
        for seq in (self.sig_model, self.col_model):
            for m in seq:
                if isinstance(m, nn.Linear):
                    ps += [m.weight, m.bias]
        return ps

    def _reflatten(self):
        ps = self._ordered()
        n = sum(p.numel() for p in ps)
        flat = torch.empty(n, device=ps[0].device, dtype=torch.float32)
        o = 0
        with torch.no_grad():
            for p in ps:
                v = flat[o:o + p.numel()].view(p.shape)
                v.copy_(p.data)
                p.data = v
                o += p.numel()
        self._flat = flat

    def _flat_params(self) -> torch.Tensor:
        flat = self._flat
        ok = flat is not None
        if ok:
            o = flat.data_ptr()
            for p in self._ordered():
                if p.data_ptr() != o or p.device != flat.device or p.dtype != torch.float32:
                    ok = False
                    break
                o += p.numel() * 4
        if not ok:
            self._reflatten()
        return self._flat

    def _grad_views(self, dflat):
        o, out = 0, []
        for p in self._ordered():
            out.append(dflat[o:o + p.numel()].view(p.shape))
            o += p.numel()
        return out

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._flat = None
        return out

    def _dims(self) -> MlpDims:
        return MlpDims(self._in0, self.d_view)

    _dp_params = _ordered

    def _dp_template(self) -> torch.Tensor:
        return self._flat_params()

    def _dp_param_views(self, buf: torch.Tensor):
        return list(zip(self._ordered(), self._grad_views(buf)))

    def _check_native(self):
        if not self._native:
            raise NotImplementedError("native MLP_3D supports num_sig=2, num_col=2, h_size=64 (the reference's configuration)")

    @staticmethod
    def _tc_operand(use_tc=None) -> int:
        """0 = fp32 CUDA-core kernels; otherwise the tensor-core operand format (ops.HBR_F16 / HBR_BF16).  use_tc: None =
        follow torch.autocast (its dtype picks the format), False, True (bf16 unless fp16 autocast is active) or a dtype."""
        if use_tc is None:
            use_tc = torch.is_autocast_enabled()
        if use_tc is False or not ops.HAS_TC:
            return 0
        return ops.tc_operand(None if use_tc is True else use_tc)

    # -- evaluation entry used by Volume_Renderer (one direction row per ray) ---------------------------------
    def field(self, feat, dirs_enc, dir_group, use_tc=None, raw=False):
        """(N,4) [rgb, density].  With use_sdf the density column is 2*sigmoid(pre-activation) - 1 (test_hash.py:59-60)
        unless raw=True."""
        self._check_native()
        out = _MlpFn.apply(feat, dirs_enc, int(dir_group), self, self._tc_operand(use_tc), *node_params(self))
        if self.use_sdf and not raw:
            out = torch.cat((out[:, :3], self._sdf_from_density(out[:, 3:4])), dim=-1)
        return out

    # -- SDF mode (test_hash.py:59-60,78-105; SURVEY 8f row 4) ------------------------------------------------
    # Composed from the path's kernels plus elementwise torch ops on the device: the kernels end the density head with
    # LeakyReLU(0.01), which is invertible, so the pre-activation the SDF head needs is recovered as d > 0 ? d : 100 d
    # (1 ulp from the true pre-activation; autograd through kernel + inverse has slope exactly 1 or 0.01 * 100).
    @staticmethod
    def _sdf_from_density(density: torch.Tensor) -> torch.Tensor:
        raw = torch.where(density > 0, density, density * 100.0)
        return 2 * torch.sigmoid(raw) - 1                                # test_hash.py:60

    def _density(self, x) -> torch.Tensor:
        """LeakyReLU(dens_vec[:, 0:1]) of the sigma net for (N, L*F+E) features, with autograd when anything needs it."""
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            if self.sdf_follows_autocast and self._tc_operand(None):
                z = torch.zeros((x.shape[0], self.d_view), device=x.device)
                return self.field(x, z, 1, use_tc=None, raw=True)[:, 3:4]       # 16-bit tensor-core kernels (whole field)
            self._check_native()
            return _DensityFn.apply(x, self, *node_params(self))
        density, _ = ops.mlp_fwd_f32(x.float().contiguous(), None, 1, self._flat_params(), self._dims(), keep_act=False)
        return density

    def forward_sdf(self, x, encoder=None):
        """test_hash.py:78-84: signed-distance-like value 2*sigmoid(.) - 1 in (-1, 1); fp32 kernels (the finite
        differences below need more than bf16)."""
        if encoder is not None:
            x = encoder(x)
        return self._sdf_from_density(self._density(x))

    def finite_difference_normals_approximator(self, x, epsilon=0.0005, encoder=None):
        """test_hash.py:86-105: central differences of forward_sdf along x, y, z at clamped positions (6 extra
        encoder + sigma-net passes)."""
        lo, hi = self.min_bound, self.max_bound
        cols = []
        for axis in range(3):
            e = torch.zeros((1, 3), device=x.device)
            e[0, axis] = epsilon
            pos = self.forward_sdf((x + e).clamp(lo, hi), encoder)[:, :1]
            neg = self.forward_sdf((x - e).clamp(lo, hi), encoder)[:, :1]
            cols.append(0.5 * (pos - neg) / epsilon)
        return torch.cat(cols, dim=-1)

    def _bounds_host(self):
        """(min_bound, max_bound) as host floats for the stencil kernel's clamp; one read-back per change of the tensors."""
        key = (self.min_bound.data_ptr(), self.min_bound._version, self.max_bound.data_ptr(), self.max_bound._version)
        if getattr(self, "_bounds_key", None) != key:
            lo = self.min_bound.detach().float().reshape(-1).cpu().tolist()
            hi = self.max_bound.detach().float().reshape(-1).cpu().tolist()
            self._bounds_val = (lo * 3 if len(lo) == 1 else lo, hi * 3 if len(hi) == 1 else hi)
            self._bounds_key = key
        return self._bounds_val

    def eikonal_norms(self, x, epsilon=0.0005, encoder=None, with_grads=False):
        """eikonal_value(finite_difference_normals_approximator(x)) (helper.py:87-89) as a 6-point stencil: one kernel forms
        the six clamped positions, ONE encoder pass and ONE density-head pass (fp32 kernels) evaluate them, one kernel turns
        the six values into 2*sigmoid - 1, the central differences and their norm -- instead of six encoder + sigma-net
        passes and ~30 elementwise launches; the backward is the mirror image (gradients reach the tables and the MLP
        through the same autograd nodes as any other encoder / field call)."""
        self._check_native()
        if not x.is_cuda:
            raise RuntimeError("MLP_3D.eikonal_norms needs CUDA tensors (there is no CPU fallback)")
        if encoder is None:
            raise ValueError("eikonal_norms takes sample POSITIONS and needs the encoder")
        x = x.detach().reshape(-1, 3)
        n = x.shape[0]
        lo, hi = self._bounds_host()
        pts = ops.sdf_stencil_points(x, float(epsilon), lo, hi)
        dens = self._density(encoder(pts.view(6 * n, 3)))
        norm, grads = ops.SdfEikonal.apply(dens.reshape(6, n), float(epsilon))
        return (norm, grads) if with_grads else norm

    def forward(self, x, viewdirs=None, mask=None):
        self._check_native()
        if not x.is_cuda:
            raise RuntimeError("MLP_3D.forward needs CUDA tensors (there is no CPU fallback)")
        if viewdirs is None:
            # the density-only branch (test_hash.py:73-77) is inference-only in the reference's callers
            density = self._density(x)
            if self.use_sdf:
                density = self._sdf_from_density(density)
            return density * mask if mask is not None else density
        out = self.field(x, viewdirs, 1)
        if mask is not None:
            out = out * mask[..., None]
        return out
