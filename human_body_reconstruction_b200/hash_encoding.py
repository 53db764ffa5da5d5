"""Drop-in for the reference's hash_encoding.py: `HashEncoder` with the same constructor, forward signature,
`Embedding_list` attribute and state_dict keys (`Embedding_list.{i}.weight`, (T,F) fp32), backed by the
sm_100a kernels in csrc/hash_grid.cu.

Storage: all L tables live in ONE contiguous (L,T,F) fp32 buffer; `Embedding_list[i].weight` are Parameter
views into it, so torch optimisers / checkpoints see the reference layout while the kernels (and the NCCL
gradient all-reduce) see a single flat tensor.  Gradients come back the same way: one fresh flat (L,T,F)
buffer per backward, handed to autograd as per-level views.
"""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import ops


class _HashEncodeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, enc, *weights):
        table = enc._flat_table()
        geom = enc._geom()
        y = ops.hash_encode_fwd(x, table, geom)
        ctx.enc = enc
        ctx.geom = geom
        ctx.table = table if ctx.needs_input_grad[0] else None     # the tables the positions' gradient is taken at
        ctx.save_for_backward(x)
        ctx.g = None
        if any(ctx.needs_input_grad[2:]):
            if enc._dp is not None:
                enc._dp.note_forward(enc)
            else:
                ctx.g = enc._zeroed_grad_async()
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        enc = ctx.enc
        L, T, F = enc.L, enc.T, enc.F
        dp = enc._dp
        # HashEncoder.position_grad: dL/dx through the trilinear weights (first order only)
        dx = ops.hash_encode_dx(x, ctx.table, ctx.geom, dy).to(x.dtype) if ctx.table is not None else None
        ctx.table = None
        if not any(ctx.needs_input_grad[2:]):       # positions only (frozen tables): no table gradient to form
            return (dx, None) + (None,) * L
        if dp is not None:
            # Data-parallel run (dist._GradExchange): accumulate into the persistent buffer of this backward pass.  The
            # last table backward of the pass runs in level chunks and publishes each one as soon as its scatter-add is
            # enqueued: that chunk's all-reduce travels over NVLink while the next chunk's scatter-add still runs.  The
            # exchange hands the reduced buffer to .grad at the end of backward; nothing is returned to autograd here.
            g, last = dp.enter_backward(enc)
            plan = dp.stream_plan(enc, L, x.shape[0]) if last else None
            if plan is not None:
                # streamed exchange (dist.PeerGradAllReduce(streamed=True)): one scatter-add launch finishing the level
                # chunks in order, one exchange launch beside it on the reducer's side stream
                ev_pre = torch.cuda.current_stream().record_event()
                ops.hash_encode_bwd_stream(x, dy[:, : L * F], ctx.geom, g, plan, dp.done)
                dp.exchange_streamed(plan, ops.hash_bwd_stream_tiles(x.shape[0]), after=(ev_pre,))
                return (dx, None) + (None,) * L
            for l0, l1 in (dp.level_chunks(enc, L, x.shape[0]) if last else [(0, L)]):
                ops.hash_encode_bwd(x, dy[:, : L * F], ctx.geom, g, l0, l1)
                if last:
                    dp.publish(enc, g[l0:l1])
            return (dx, None) + (None,) * L
        if ctx.g is not None:
            g, ev = ctx.g
            ctx.g = None
            torch.cuda.current_stream().wait_event(ev)
        else:
            g = torch.zeros((L, T, F), device=dy.device, dtype=torch.float32)
        ops.hash_encode_bwd(x, dy[:, : L * F], ctx.geom, g, 0, L)
        # no gradient w.r.t. x unless position_grad is set: the reference detaches the interpolation weights
        # (hash_encoding.py:160)
        return (dx, None) + tuple(g[i] for i in range(L))


class HashEncoder(nn.Module):
    """hash_encoding.py:5-170.  Only dim == 3 has a CUDA implementation (dim == 2 serves the reference's
    broken 2-D image demo, test_hash.py:108-205, which is out of scope).

    `position_grad` (default False, the reference's behaviour: positions are detached): when True and x.requires_grad,
    forward keeps x in the graph and backward returns dL/dx from hbr_hash_encode_dx -- the trilinear weights
    differentiated at the forward's cells, first order only (once_differentiable).  So
    torch.autograd.grad(nerf(encoder(x))[:, 0].sum(), x) is the density's spatial gradient.  The fused ray routes of
    Volume_Renderer form the sample positions inside their kernels and never call this forward: they have no position
    gradient whatever the flag says."""

    def __init__(self, N_max, N_min, L, E=0, T=2 ** 14, F=2, dim=2, mu=None, sigma=None, device=None):
        super().__init__()
        if device is None:
            device = "cuda" if torch.cuda.is_available() else "cpu"
        self.device = device
        # hash_encoding.py:11-13 -- CPU scalars, evaluated exactly like the reference so the per-level
        # scales N_min*b**i are bit-identical (they are NOT floored and are fp32)
        self.N_max = torch.tensor(N_max)
        self.N_min = torch.tensor(N_min)
        self.b = torch.exp((torch.log(self.N_max) - torch.log(self.N_min)) / (L - 1))
        self.L, self.F, self.T, self.E, self.dim = int(L), int(F), int(T), int(E), int(dim)
        self.sigma = 1 if sigma is None else sigma.to(self.device)
        self.mu = 0 if mu is None else mu
        tables = []
        for _ in range(self.L):
            emb = nn.Embedding(self.T, self.F, sparse=False)          # same RNG draws as the reference (:31-32)
            nn.init.uniform_(emb.weight, a=-1e-4, b=1e-4)
            tables.append(emb)
        self.Embedding_list = nn.ModuleList(tables)
        self._scales = [float((self.N_min * self.b ** i).to(torch.float32)) for i in range(self.L)]   # :153
        self._host_geom = None
        self._side = None
        self._dp = None               # the data-parallel gradient exchange attached to this module (dist._GradExchange)
        self._flat = None
        self.position_grad = False    # see the class docstring
        self._reflatten()

    # -- flat storage ------------------------------------------------------------------------------------
    def _reflatten(self):
        ws = [e.weight for e in self.Embedding_list]
        flat = torch.empty((self.L, self.T, self.F), device=ws[0].device, dtype=torch.float32)
        with torch.no_grad():
            for i, w in enumerate(ws):
                flat[i].copy_(w.data)
                w.data = flat[i]
        self._flat = flat

    def _flat_table(self) -> torch.Tensor:
        """The (L,T,F) buffer all level tables are views of (re-established after .to()/load of foreign storage)."""
        flat = self._flat
        step = self.T * self.F * 4
        ok = flat is not None
        if ok:
            base = flat.data_ptr()
            for i, e in enumerate(self.Embedding_list):
                w = e.weight
                if w.data_ptr() != base + i * step or w.device != flat.device or w.dtype != torch.float32:
                    ok = False
                    break
        if not ok:
            self._reflatten()
        return self._flat

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._flat = None
        self._host_geom = None
        return out

    def _geom(self):
        if self._host_geom is None:
            mu = self.mu
            if torch.is_tensor(mu):
                mu = [float(v) for v in mu.detach().reshape(-1).cpu()]
                if len(mu) == 1:
                    mu = mu * 3
            else:
                mu = [float(mu)] * 3
            sigma = float(self.sigma.detach().cpu()) if torch.is_tensor(self.sigma) else float(self.sigma)
            self._host_geom = ops.make_geom(mu, sigma, self._scales, self.L, self.F, self.T, self.E)
        return self._host_geom

    def _zeroed_grad_async(self):
        """A zero-filled (L,T,F) gradient buffer whose 64 MiB memset runs on a side stream, i.e. concurrently with the
        forward kernels instead of in front of the scatter-add.  Returns (buffer, event the consumer must wait for)."""
        dev = self._flat.device
        cur = torch.cuda.current_stream(dev)
        side = self._side
        if side is None or side.device != dev:
            side = self._side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            g = torch.zeros((self.L, self.T, self.F), device=dev, dtype=torch.float32)
            ev = side.record_event()
        g.record_stream(cur)
        return g, ev

    # -- data-parallel gradient exchange (dist._GradExchange) ---------------------------------------------------
    def _dp_template(self) -> torch.Tensor:
        return self._flat_table()

    def _dp_param_views(self, buf: torch.Tensor):
        return [(e.weight, buf[i]) for i, e in enumerate(self.Embedding_list)]

    def level_scales(self):
        return list(self._scales)

    def hash_indices(self, x):
        """(L,N,8) int32 table indices and (L,N,8) weights -- the values hash_encoding.py:161-164 computes."""
        return ops.hash_indices(x, self._geom())

    def forward(self, x, aux=None):
        assert x.shape[-1] == self.dim
        if self.dim != 3:
            raise NotImplementedError("the sm_100a HashEncoder implements dim=3 only")
        if not x.is_cuda:
            raise RuntimeError("HashEncoder.forward needs CUDA tensors (there is no CPU fallback)")
        if x.dim() != 2:
            raise ValueError("x must be (N,3)")
        if x.dtype not in (torch.float32, torch.float16):
            x = x.float()
        table = self._flat_table()
        if table.device != x.device:
            raise RuntimeError(f"encoder tables are on {table.device}, x on {x.device}")
        weights = [e.weight for e in self.Embedding_list]
        if not torch.is_grad_enabled():
            # needs_input_grad follows requires_grad, not the grad mode: under no_grad the node would still zero a table
            # gradient buffer that no backward ever reads
            weights = [w.detach() for w in weights]
        keep = getattr(self, "position_grad", False) and x.requires_grad and torch.is_grad_enabled()
        return _HashEncodeFn.apply(x if keep else x.detach(), self, *weights)
