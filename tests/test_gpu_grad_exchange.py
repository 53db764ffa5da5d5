"""The modules' side of the gradient exchange (dist.node_params / dist.ParamGrad) on one device, with an exchange attached
at world size 1, on every route of a training step: the fp32 modules (_HashEncodeFn, _MlpFn), the autocast modules
(chain_field=False), the chained autocast node (_FieldRaysFn, fused scatter on and off), the fused field (_FieldFn), the
compacted samples (_FieldCompactFn) and native SDF mode with its eikonal term (_DensityFn).  Each route gives the gradients
it gives without an exchange, every backward closes exactly one session with no node left expected, frozen tables get no
gradient, and a no_grad render counts no node."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
EXCHANGES = ["nccl-1", "nccl-4", "peer-launch", "peer-launch-lm", "peer-stream", "peer-stream-lm"]
# (route, hierarchical): SDF mode's native route is single-pass only
ROUTES = [(r, h) for r in ("fp32", "amp-modules", "amp-chained", "amp-chained-unfused", "fuse-field", "compact")
          for h in (False, True)] + [("sdf-fp32", False), ("sdf-amp", False)]


def _build(sdf):
    import human_body_reconstruction_b200 as h
    torch.manual_seed(0)
    mu, maxb = torch.tensor([-4.27, -4.31, -3.95]), torch.tensor([4.28, 4.27, 2.37])
    sigma = ((maxb - mu) ** 2).sum().sqrt()
    enc = h.HashEncoder(N_min=16, N_max=2048.0, L=16, F=2, T=2 ** 14, dim=3, mu=mu.to(DEV), sigma=sigma.to(DEV))
    with torch.no_grad():
        for e in enc.Embedding_list:
            e.weight.mul_(5e3)
    mlp = h.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=maxb, min_bound=mu)
    enc, mlp = enc.to(DEV), mlp.to(DEV)
    var = h.helper.VarModel().to(DEV) if sdf else None
    vr = h.Volume_Renderer(H=8, W=8, K=torch.eye(3), near=torch.tensor(2.0), far=torch.tensor(6.0), device=DEV,
                           Pos_encode=enc, Dir_encode=h.PositionalEncoder(3, 4), max_dim=64, sigma_val=sigma, mu=mu,
                           use_sdf=sdf, var_model=var)
    return enc, mlp, vr


def _batch():
    g = torch.Generator().manual_seed(11)
    R = 256
    ro = torch.tensor([[0.2, -0.1, 4.0]]).repeat(R, 1) + 0.05 * torch.randn(R, 3, generator=g)
    rd = torch.nn.functional.normalize(-ro + 0.5 * torch.randn(R, 3, generator=g), dim=-1)
    return (ro, rd, 1 + 0.2 * torch.rand(R, 1, generator=g), torch.rand(R, 3, generator=g), torch.rand(R, 32, generator=g),
            torch.linspace(2.0, 6.0, 32), torch.rand(32, generator=g))


def _render(mlp, vr, amp, hier):
    import human_body_reconstruction_b200 as h
    ro, rd, dn, gt, u, t, u_cand = (v.to(DEV) for v in _batch())
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        Cr, Cf, norm = vr.vol_render(mlp, rd, ro, num_samples=32, t=t, dir_norm=dn, hierarchical=hier, _u=u, _u_cand=u_cand)
        if not torch.is_grad_enabled():
            return None
        loss = torch.nn.functional.mse_loss(Cr, gt) + torch.nn.functional.mse_loss(Cf, gt)
        if norm is not None:
            loss = loss + 0.1 * h.helper.eikonal_loss(norm)
    return loss


def _grads(enc, mlp, vr, amp, hier):
    """One backward: (table gradient (L,T,F) or None, flat MLP gradient), copied."""
    for p in list(enc.parameters()) + list(mlp.parameters()):
        p.grad = None
    _render(mlp, vr, amp, hier).backward()
    torch.cuda.synchronize()        # world 1: the end of backward does not join the exchange's side stream
    tab = [e.weight.grad for e in enc.Embedding_list]
    return (None if tab[0] is None else torch.stack(tab).clone(),
            torch.cat([p.grad.reshape(-1) for p in mlp.parameters()]).clone())


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("route,hier", ROUTES)
@pytest.mark.parametrize("kind", EXCHANGES)
def test_exchange_at_world_one(kind, route, hier, monkeypatch):
    from human_body_reconstruction_b200 import dist as hdist
    from human_body_reconstruction_b200 import vol_renderer as vrm
    enc, mlp, vr = _build(route.startswith("sdf"))
    amp = route != "fp32" and route != "sdf-fp32"
    vr.chain_field = route != "amp-modules"
    vr.fuse_field = route == "fuse-field"
    monkeypatch.setattr(vrm, "FUSE_SCATTER", route != "amp-chained-unfused")
    monkeypatch.setattr(vrm, "STREAM_LEVEL_MAJOR", kind.endswith("-lm"))
    if route == "compact":
        vr.compact = True
        i = torch.arange(vr.grid_size, device=DEV)
        vr.bool_grid[...] = (i[:, None, None] + i[None, :, None] + i[None, None, :]) % 2 == 0     # half the cells
    # fp32 and autocast: test_gpu_multi.py's bars (atomics in the scatter-add); SDF mode: its bar there too -- the stencil's
    # +-1/(2 eps) coefficients land on the same table entries with opposite signs and amplify the summation-order noise
    tol = 2e-3 if route.startswith("sdf") else (1e-4 if amp else 1e-5)
    want_tab, want_mlp = _grads(enc, mlp, vr, amp, hier)
    if kind.startswith("nccl"):
        red = hdist.GradAllReduce(enc, mlp, chunks=int(kind[-1]))
    else:
        red = hdist.PeerGradAllReduce(enc, mlp, overlap=True, chunks=4, streamed=kind.startswith("peer-stream"))
    try:
        for _ in range(2):                                   # twice through the same persistent buffers
            sessions = red.sessions
            tab, gm = _grads(enc, mlp, vr, amp, hier)
            assert red.sessions == sessions + 1 and not any(red._fwd.values()), red._fwd
            assert _rel(tab, want_tab) < tol and _rel(gm, want_mlp) < tol, (_rel(tab, want_tab), _rel(gm, want_mlp))
        for e in enc.Embedding_list:                         # frozen tables
            e.weight.requires_grad_(False)
        tab, gm = _grads(enc, mlp, vr, amp, hier)
        assert tab is None and _rel(gm, want_mlp) < tol
        assert not any(red._fwd.values()), red._fwd
        for e in enc.Embedding_list:
            e.weight.requires_grad_(True)
        sessions = red.sessions
        with torch.no_grad():
            _render(mlp, vr, amp, hier)
        assert not any(red._fwd.values()) and red.sessions == sessions, red._fwd
    finally:
        red.remove()
        if hasattr(red, "region"):
            torch.cuda.synchronize()
            red.region.close()
