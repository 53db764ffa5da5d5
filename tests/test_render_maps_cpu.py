"""CPU: depth / opacity maps of the compositor and Volume_Renderer.render / render_view without a GPU.
  * the closed-form backward with depth and opacity gradients (maps_oracle.composite_maps_bwd, the derivation
    hbr_composite_maps_bwd implements) == float64 autograd of port.composite, for shared and per-ray depths, across the
    -10 density clamp;
  * render and render_view raise RuntimeError naming CUDA on a host without a GPU (there is no CPU fallback)."""
import pytest
import torch
from hypothesis import given, settings, strategies as st

import maps_oracle
from oracle import port

SET = settings(max_examples=60, deadline=None, derandomize=True, database=None)


@SET
@given(st.integers(0, 2 ** 31 - 1), st.integers(2, 40), st.booleans())
def test_maps_closed_form_backward_matches_autograd(seed, S, per_ray):
    g = torch.Generator().manual_seed(seed)
    R = 5
    shape = (R, S) if per_ray else (S,)
    t = torch.sort(torch.rand(*shape, generator=g, dtype=torch.float64) * 4 + 2, dim=-1).values
    rgb = torch.rand(R, S, 3, generator=g, dtype=torch.float64).requires_grad_(True)
    sigma = (torch.randn(R, S, generator=g, dtype=torch.float64) * 8).requires_grad_(True)   # crosses the -10 clamp
    dn = 1 + torch.rand(R, 1, generator=g, dtype=torch.float64)
    C, w = port.composite(t, rgb, sigma, dn)
    depth = (w * (t[None, :] if t.dim() == 1 else t)).sum(-1)
    opacity = w.sum(-1)
    C2, w2, D2, A2 = maps_oracle.composite_maps(t, rgb.detach(), sigma.detach(), dn)
    assert torch.equal(C2, C.detach()) and torch.equal(w2, w.detach())
    assert torch.allclose(D2, depth.detach(), rtol=1e-12, atol=0) and torch.allclose(A2, opacity.detach(), rtol=1e-12, atol=0)
    gC = torch.randn(R, 3, generator=g, dtype=torch.float64)
    gD = torch.randn(R, generator=g, dtype=torch.float64)
    gA = torch.randn(R, generator=g, dtype=torch.float64)
    ((C * gC).sum() + (depth * gD).sum() + (opacity * gA).sum()).backward()
    drgb, dsig = maps_oracle.composite_maps_bwd(t, rgb.detach(), sigma.detach(), dn, gC, gD, gA)
    assert torch.allclose(drgb, rgb.grad, rtol=1e-9, atol=1e-9)
    scale = sigma.grad.abs().max(dim=-1, keepdim=True).values + 1.0      # per ray: suffix sums cancel
    assert bool(((dsig - sigma.grad).abs() <= 1e-8 * scale).all())
    assert bool((dsig[sigma.detach() < -10] == 0).all())
    # gD = gA = 0 is the colour-only backward
    z = torch.zeros(R, dtype=torch.float64)
    d0 = maps_oracle.composite_maps_bwd(t, rgb.detach(), sigma.detach(), dn, gC, z, z)
    ref = port.composite_bwd(t, rgb.detach(), sigma.detach(), dn, gC)
    assert torch.equal(d0[0], ref[0]) and torch.equal(d0[1], ref[1])


def _renderer():
    import human_body_reconstruction_b200 as h
    enc = h.HashEncoder(N_min=16, N_max=512.0, L=16, F=2, T=64, dim=3, mu=torch.zeros(3), sigma=torch.tensor(1.0), device="cpu")
    vr = h.Volume_Renderer(H=4, W=6, K=torch.eye(3), near=2.0, far=6.0, device="cpu", Pos_encode=enc,
                           Dir_encode=h.PositionalEncoder(3, 4), max_dim=16)
    mlp = h.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=torch.ones(3), min_bound=-torch.ones(3))
    return vr, mlp


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour on a host without a GPU")
def test_render_and_render_view_need_cuda():
    vr, mlp = _renderer()
    with pytest.raises(RuntimeError, match="CUDA"):
        vr.render(mlp, torch.randn(3, 3), torch.zeros(3, 3), num_samples=8, t=torch.linspace(2, 6, 8), hierarchical=False)
    with pytest.raises(RuntimeError, match="CUDA"):
        vr.render_view(mlp, torch.eye(4), num_samples=8)
