"""GPU: depth and opacity maps (hbr_composite_maps_fwd/bwd, ops.CompositeMapsPacked) and the rendering entry points built
on them (Volume_Renderer.render, Volume_Renderer.render_view).

  * kernel level, against float64 autograd of oracle.port.composite: every input form of the compositor (shared / per-ray
    depths, dir_norm tensor / scalar, mask, compacted rowmap), 1e-5 relative to the magnitude of each ray's terms; C and w
    bit-identical to hbr_composite_fwd; with gD = gA = 0 the gradients bit-identical to hbr_composite_bwd; early ray
    termination changes nothing for sigma >= 0;
  * render: colours bit-identical to vol_render on every route, maps and their gradients against the oracle; the native
    SDF route against float64 autograd of port.composite_sdf;
  * render_view: a hand loop of ray_gen + render, the oracle's get_od + vol_render, independence of the chunk size, memory
    bounded by the chunk, nothing allocated for table gradients."""
import pytest
import torch

from conftest import capture_fine_sampling, load_golden, mlp_params
import maps_oracle
from oracle import port

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def check_rows(a, b, tol=1e-5):
    a, b = a.detach().double().cpu().flatten(1), b.detach().double().cpu().flatten(1)
    err = (a - b).norm(dim=1)
    assert (err <= tol * b.norm(dim=1) + 1e-12).all(), float((err / (b.norm(dim=1) + 1e-30)).max())


def check_maps(D, A, D_ref, A_ref, w_ref, t_ref, tol=1e-5):
    """Relative to the magnitude of the terms of each ray: negative densities make weights cancel (as check_composite in
    test_gpu_parity does for the colour)."""
    D, A = D.detach().double().cpu(), A.detach().double().cpu()
    tt = t_ref[None, :] if t_ref.dim() == 1 else t_ref
    sD = (w_ref.abs() * tt.abs()).sum(-1)
    sA = w_ref.abs().sum(-1)
    assert ((D - D_ref).abs() <= tol * sD + 1e-6).all(), float(((D - D_ref).abs() / (sD + 1e-30)).max())
    assert ((A - A_ref).abs() <= tol * sA + 1e-7).all(), float(((A - A_ref).abs() / (sA + 1e-30)).max())


# ---- kernel level ----------------------------------------------------------------------------------------------------
def _case(S, tkind, dnkind, form, seed):
    """R rays of S samples -> (t, out4 (R*S,4), dir_norm, mask or None, live (R*S) bool) on the host, fp32.  Per-ray depths
    are shaped like the fine pass's (R, 2S), capped at the compositor's 1024 samples."""
    g = torch.Generator().manual_seed(seed)
    R = 45
    Se = min(2 * S, 1024) if tkind == "perray" else S
    shape = (R, Se) if tkind == "perray" else (Se,)
    t = torch.sort(2 + 4 * torch.rand(*shape, generator=g), dim=-1).values
    out4 = torch.rand(R * Se, 4, generator=g)
    out4[:, 3] = torch.randn(R * Se, generator=g) * 3                     # LeakyReLU-like: some negative densities
    dn = (1 + torch.rand(R, 1, generator=g)) if dnkind == "tensor" else 1.3
    live = torch.ones(R * Se, dtype=torch.bool) if form == "plain" else torch.rand(R * Se, generator=g) > 0.35
    return R, Se, t, out4, dn, live


def _oracle64(R, S, t, out4, dn, live, gC, gD, gA):
    """float64 autograd of port.composite with depth / opacity formed from its weights; skipped samples are rgb = sigma = 0
    (vol_renderer.py:211-216).  Returns (C, w, D, A, d out4 (R*S,4) on the live samples, 0 elsewhere)."""
    o = (out4.double() * live[:, None].double()).requires_grad_()
    dn64 = dn.double() if torch.is_tensor(dn) else dn
    C, w, D, A = maps_oracle.composite_maps(t.double(), o[:, :3].reshape(R, S, 3), o[:, 3].reshape(R, S), dn64)
    ((C * gC.double()).sum() + (D * gD.double()).sum() + (A * gA.double()).sum()).backward()
    return C.detach(), w.detach(), D.detach(), A.detach(), o.grad * live[:, None].double()


@pytest.mark.parametrize("form", ["plain", "mask", "rowmap"])
@pytest.mark.parametrize("dnkind", ["tensor", "scalar"])
@pytest.mark.parametrize("tkind", ["shared", "perray"])
@pytest.mark.parametrize("S", [7, 32, 100, 128, 256, 1024])
def test_maps_kernels_against_float64(S, tkind, dnkind, form):
    from human_body_reconstruction_b200 import ops
    R, S, t, out4, dn, live = _case(S, tkind, dnkind, form, 1000 + S)
    g = torch.Generator().manual_seed(S)
    gC, gD, gA = torch.randn(R, 3, generator=g), torch.randn(R, generator=g), torch.randn(R, generator=g)
    C_ref, w_ref, D_ref, A_ref, d_ref = _oracle64(R, S, t, out4, dn, live, gC, gD, gA)

    td = t.to(DEV)
    dnd = dn.to(DEV) if torch.is_tensor(dn) else dn
    mask, rowmap = None, None
    if form == "mask":
        mask = live.to(DEV)
        o_in = out4.to(DEV)
    elif form == "rowmap":
        rows = torch.cumsum(live.to(torch.int64), 0) - 1
        rowmap = torch.where(live, rows, torch.full_like(rows, -1)).to(torch.int32).to(DEV)
        o_in = out4[live].to(DEV)                                          # the compacted list
    else:
        o_in = out4.to(DEV)
    o = o_in.clone().requires_grad_()
    C, w, D, A = ops.CompositeMapsPacked.apply(o, td, dnd, mask, R, S, 0.0, rowmap)
    scale = (w_ref.abs()[..., None] * (out4[:, :3] * live[:, None]).reshape(R, S, 3).double().abs()).sum(1)
    assert ((C.detach().cpu().double() - C_ref).abs() <= 1e-5 * scale + 1e-6).all()
    check_maps(D, A, D_ref, A_ref, w_ref, t.double())

    # C and w are those of hbr_composite_fwd, bit for bit
    C0, w0 = ops.CompositePacked.apply(o_in, td, dnd, mask, R, S, 0.0, rowmap)
    assert torch.equal(C.detach(), C0) and torch.equal(w, w0)

    # random gC, gD, gA: float64 autograd, norm-wise per ray
    (C * gC.to(DEV)).sum().add((D * gD.to(DEV)).sum()).add((A * gA.to(DEV)).sum()).backward()
    grad = torch.zeros(R * S, 4, device=DEV)
    if form == "rowmap":
        grad[live.to(DEV)] = o.grad
    else:
        grad = o.grad * live.to(DEV)[:, None]
    check_rows(grad.view(R, S * 4), d_ref.view(R, S * 4))

    # gD = gA = 0: the gradients of hbr_composite_bwd, bit for bit
    zc = torch.zeros(R, device=DEV)
    g0 = torch.empty_like(o_in)
    g1 = torch.empty_like(o_in)
    ops.composite_maps_bwd(td, o_in, 4, o_in[:, 3:], 4, dnd, mask, R, S, gC.to(DEV), zc, zc, g0, 4, g0[:, 3:], 4, rowmap=rowmap)
    ops.composite_bwd(td, o_in, 4, o_in[:, 3:], 4, dnd, mask, R, S, gC.to(DEV), g1, 4, g1[:, 3:], 4, rowmap=rowmap)
    n = int(live.sum()) if form == "rowmap" else R * S
    assert torch.equal(g0[:n], g1[:n])
    # NULL gradients read as 0
    g2 = torch.empty_like(o_in)
    ops.composite_maps_bwd(td, o_in, 4, o_in[:, 3:], 4, dnd, mask, R, S, gC.to(DEV), None, None, g2, 4, g2[:, 3:], 4, rowmap=rowmap)
    assert torch.equal(g2[:n], g1[:n])


def test_maps_with_early_ray_termination_are_exact():
    """sigma >= 0: the skipped chunks had transmittance exactly 0, so maps and gradients are bit-identical with and without
    early ray termination at ops.ERT_TAU, and the tail really was skipped."""
    from human_body_reconstruction_b200 import ops
    torch.manual_seed(4)
    R, S = 300, 256
    t = torch.sort(2 + 4 * torch.rand(R, S), dim=-1).values.to(DEV)
    gC, gD, gA = torch.randn(R, 3, device=DEV), torch.randn(R, device=DEV), torch.randn(R, device=DEV)
    for dense in (False, True):
        out4 = torch.rand(R * S, 4, device=DEV)
        out4[:, 3] *= 4000.0 if dense else 3.0
        res = []
        for tau in (0.0, ops.ERT_TAU):
            o = out4.clone().requires_grad_()
            C, w, D, A = ops.CompositeMapsPacked.apply(o, t, 1.0, None, R, S, tau)
            ((C * gC).sum() + (D * gD).sum() + (A * gA).sum()).backward()
            res.append((C.detach(), w, D.detach(), A.detach(), o.grad.clone()))
        for a, b in zip(*res):
            assert torch.equal(a, b)
        if dense:
            assert float((res[1][1][:, 64:] == 0).float().mean()) == 1.0


# ---- Volume_Renderer.render ------------------------------------------------------------------------------------------
def _build(g, max_dim=64, H=8, W=8, K=None):
    import human_body_reconstruction_b200 as h
    L, T, F = g["tables"].shape
    enc = h.HashEncoder(N_min=16, N_max=2048.0, L=L, F=F, T=T, dim=3, mu=g["mu"].to(DEV), sigma=g["sigma"].to(DEV))
    enc.load_state_dict({f"Embedding_list.{i}.weight": g["tables"][i] for i in range(L)})
    enc = enc.to(DEV)
    mlp = h.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=torch.ones(3), min_bound=-torch.ones(3))
    mlp.load_state_dict(mlp_params(g, "mlp__"))
    mlp = mlp.to(DEV)
    vr = h.Volume_Renderer(H=H, W=W, K=torch.eye(3) if K is None else K, near=torch.tensor(float(g["near"])),
                           far=torch.tensor(float(g["far"])), device=DEV, Pos_encode=enc, Dir_encode=h.PositionalEncoder(3, 4),
                           max_dim=max_dim, sigma_val=g["sigma"], mu=g["mu"])
    return vr, enc, mlp


ROUTES = [
    # (name, hierarchical, max_points, autocast dtype, occupancy, compact, ert)
    ("fp32", False, 1 << 26, None, 1.0, False, False),
    ("fp32-hier", True, 1 << 26, None, 1.0, False, False),
    ("fp32-hier-chunked", True, 24 * 7 * 3, None, 1.0, False, False),
    ("fp32-chunked", False, 24 * 7, None, 1.0, False, False),
    ("fp32-masked", False, 1 << 26, None, 0.6, False, False),
    ("bf16-chained-hier", True, 1 << 26, torch.bfloat16, 1.0, False, False),
    ("f16-chained-hier-chunked", True, 24 * 5 * 3, torch.float16, 1.0, False, False),
    ("bf16-masked", False, 1 << 26, torch.bfloat16, 0.6, False, False),
    ("bf16-compact", False, 1 << 26, torch.bfloat16, 0.6, True, False),
    ("bf16-compact-hier", True, 1 << 26, torch.bfloat16, 0.6, True, False),
    ("fp32-ert-hier", True, 1 << 26, None, 1.0, False, True),
]


@pytest.mark.parametrize("route", ROUTES, ids=[r[0] for r in ROUTES])
def test_render_colours_equal_vol_render(route):
    from human_body_reconstruction_b200 import _lib
    name, hier, max_points, amp, occ, compact, ert = route
    g = load_golden("volrender.npz")
    vr, enc, mlp = _build(g)
    vr.max_points, vr.compact, vr.ert = max_points, compact, ert
    if occ < 1.0:
        gen = torch.Generator().manual_seed(7)
        vr.bool_grid[...] = (torch.rand(vr.bool_grid.shape, generator=gen) < occ).to(DEV)
    args = (mlp, g["rays_d"].to(DEV), g["rays_o"].to(DEV))
    kw = dict(num_samples=24, dir_norm=g["dir_norm"].to(DEV), hierarchical=hier)
    res = []
    for fn in ("vol_render", "render"):
        torch.manual_seed(5)
        _lib.STATS.reset()
        with torch.autocast("cuda", dtype=amp or torch.bfloat16, enabled=amp is not None):
            out = getattr(vr, fn)(*args, **kw)
        res.append((out, dict(_lib.STATS.calls)))
    (Cr, Cf, _), calls_v = res[0]
    out, calls_r = res[1]
    assert torch.equal(out.rgb_coarse, Cr) and torch.equal(out.rgb_fine, Cf)
    assert out.depth_coarse.shape == (Cr.shape[0],) and out.opacity_fine.shape == (Cr.shape[0],)
    if not hier:
        assert torch.equal(out.depth_fine, out.depth_coarse) and torch.equal(out.opacity_fine, out.opacity_coarse)
    # the same launches, the compositor swapped for its maps form
    swap = {"hbr_composite_fwd": "hbr_composite_maps_fwd"}
    assert {swap.get(k, k): v for k, v in calls_v.items()} == calls_r
    assert ("hbr_compact_samples" in calls_r) == compact


def _oracle_maps(pr, tb, g, t, dn, rays_o, rays_d):
    R, S = rays_o.shape[0], t.shape[-1]
    pts = port.ray_points(rays_o, rays_d, t).reshape(-1, 3)
    dirs = port.dir_encode(rays_d[:, None, :].repeat(1, S, 1).reshape(-1, 3), 4)
    out = port.mlp_forward(pr, port.hash_encode(pts, tb, g["mu"], g["sigma"], g["scales"]), dirs)
    return maps_oracle.composite_maps(t, out[:, 0:3].reshape(R, S, 3), out[:, 3].reshape(R, S), dn)


def _mask_loss(depth, opacity, m):
    """depth.sum() + binary cross-entropy of the opacity against a person mask (written out: the opacity is clamped into
    (0, 1) first, the way a mask loss on a LeakyReLU field has to be)."""
    a = opacity.clamp(1e-6, 1 - 1e-6)
    return depth.sum() - (m * torch.log(a) + (1 - m) * torch.log(1 - a)).mean()


@pytest.mark.parametrize("hier", [False, True])
def test_render_maps_and_gradients_match_oracle(hier):
    """fp32 kernels: depth and opacity against the oracle on the same t / t_fine; gradients of a depth + mask loss reaching
    the tables and the MLP within the tolerances of the vol_render gradient tests (1e-5 tables, 2e-5 MLP)."""
    g = load_golden("volrender.npz")
    vr, enc, mlp = _build(g)
    S = 24
    t = port.strat_t(g["near"], g["far"], S, g["coarse__u_t"])
    R = g["rays_o"].shape[0]
    m = (torch.arange(R) % 3 == 0).float()
    torch.manual_seed(3)
    with capture_fine_sampling() as rec:
        out = vr.render(mlp, g["rays_d"].to(DEV), g["rays_o"].to(DEV), num_samples=S, t=t.to(DEV), dir_norm=g["dir_norm"].to(DEV),
                        hierarchical=hier)
    loss = _mask_loss(out.depth_coarse, out.opacity_coarse, m.to(DEV))
    if hier:
        loss = loss + _mask_loss(out.depth_fine, out.opacity_fine, m.to(DEV))
    loss.backward()

    tb = g["tables"].clone().requires_grad_()
    pr = {k: v.clone().requires_grad_() for k, v in mlp_params(g, "mlp__").items()}
    Cr_o, w_o, Dr_o, Ar_o = _oracle_maps(pr, tb, g, t, g["dir_norm"], g["rays_o"], g["rays_d"])
    assert torch.allclose(out.rgb_coarse.detach().cpu(), Cr_o.detach(), rtol=1e-5, atol=1e-6)
    check_maps(out.depth_coarse, out.opacity_coarse, Dr_o.detach().double(), Ar_o.detach().double(), w_o.detach().double(), t.double())
    lo = _mask_loss(Dr_o, Ar_o, m)
    if hier:
        tf = rec["t_fine"].cpu()
        Cf_o, wf_o, Df_o, Af_o = _oracle_maps(pr, tb, g, tf, g["dir_norm"], g["rays_o"], g["rays_d"])
        assert torch.allclose(out.rgb_fine.detach().cpu(), Cf_o.detach(), rtol=1e-5, atol=1e-6)
        check_maps(out.depth_fine, out.opacity_fine, Df_o.detach().double(), Af_o.detach().double(), wf_o.detach().double(),
                   tf.double())
        lo = lo + _mask_loss(Df_o, Af_o, m)
    lo.backward()
    assert abs(float(loss.detach()) - float(lo.detach())) <= 1e-5 * abs(float(lo.detach())) + 1e-6
    assert rel(torch.stack([e.weight.grad for e in enc.Embedding_list]), tb.grad) < 1e-5
    for k, p in mlp.named_parameters():
        assert rel(p.grad, pr[k].grad) < 2e-5, k


def test_render_needs_the_native_modules():
    g = load_golden("volrender.npz")
    vr, enc, mlp = _build(g)
    with pytest.raises(TypeError):
        vr.render(lambda x, d: mlp(x, d), g["rays_d"].to(DEV), g["rays_o"].to(DEV), num_samples=8, hierarchical=False)


def test_render_sdf_route_maps_and_gradients():
    """Native SDF route: colours equal vol_render's; the maps come from the weights hbr_composite_sdf_fwd returns and their
    gradients (including dL/db) go through hbr_composite_sdf_bwd's weight gradient -- against float64 autograd of
    port.composite_sdf on the same field output."""
    import human_body_reconstruction_b200 as h
    g = load_golden("sdf.npz")
    L, T, F = g["tables"].shape
    enc = h.HashEncoder(N_min=16, N_max=512.0, L=L, F=F, T=T, dim=3, mu=g["mu"].to(DEV), sigma=g["sigma"].to(DEV))
    enc.load_state_dict({f"Embedding_list.{i}.weight": g["tables"][i] for i in range(L)})
    mlp = h.MLP_3D(num_sig=2, num_col=2, L=L, F=F, d_view=24, use_sdf=True, max_bound=g["max_bound"], min_bound=g["min_bound"])
    mlp.load_state_dict(mlp_params(g, "mlp__"))
    var = h.helper.VarModel().to(DEV)
    with torch.no_grad():
        var.b.fill_(float(g["b"]))
    enc, mlp = enc.to(DEV), mlp.to(DEV)
    vr = h.Volume_Renderer(H=8, W=8, K=torch.eye(3), near=torch.tensor(2.0), far=torch.tensor(6.0), device=DEV, Pos_encode=enc,
                           Dir_encode=h.PositionalEncoder(3, 4), max_dim=64, sigma_val=g["sigma"], mu=g["mu"], use_sdf=True,
                           var_model=var)
    rd, ro, t = g["rays_d"].to(DEV), g["rays_o"].to(DEV), g["t"].to(DEV)
    R, S = ro.shape[0], t.shape[0]
    Cr, _, norm = vr.vol_render(mlp, rd, ro, num_samples=S, t=t, dir_norm=g["dir_norm"].to(DEV), hierarchical=False)
    out = vr.render(mlp, rd, ro, num_samples=S, t=t, dir_norm=g["dir_norm"].to(DEV), hierarchical=False)
    assert torch.equal(out.rgb_coarse, Cr) and torch.equal(out.norm, norm) and out.rgb_fine is out.rgb_coarse
    gD, gA = torch.randn(R, device=DEV), torch.randn(R, device=DEV)
    var.b.grad = None
    ((out.depth_coarse * gD).sum() + (out.opacity_coarse * gA).sum()).backward()
    db = float(var.b.grad)

    # the same field output, composited in float64
    with torch.no_grad():
        dir_enc = vr.Dir_encode(rd.float().contiguous())
        pts = h.ops.ray_points(ro, rd, t).view(-1, 3)
        out4 = mlp.field(enc(pts), dir_enc, S, raw=True).double().cpu()
    dens = out4[:, 3]
    sdf = (2 * torch.sigmoid(torch.where(dens > 0, dens, dens * 100.0)) - 1).reshape(R, S)   # from_density, as the kernel
    b64 = torch.tensor(float(g["b"]), dtype=torch.float64, requires_grad=True)
    _, w = port.composite_sdf(out4[:, :3].reshape(R, S, 3), sdf, b64)
    w = w[..., 0]
    D_ref, A_ref = (w * g["t"].double()).sum(-1), w.sum(-1)
    assert rel(out.depth_coarse, D_ref) < 5e-5 and rel(out.opacity_coarse, A_ref) < 5e-5
    ((D_ref * gD.double().cpu()).sum() + (A_ref * gA.double().cpu()).sum()).backward()
    assert abs(db - float(b64.grad)) < 2e-4 * abs(float(b64.grad)) + 2e-5


# ---- Volume_Renderer.render_view -------------------------------------------------------------------------------------
def _view_setup(H=24, W=32, V=2):
    import bench
    g = load_golden("volrender.npz")
    K = bench.intrinsics(H, W)
    vr, enc, mlp = _build(g, H=H, W=W, K=K)
    c2w = bench.make_cameras(V, 3)
    return g, vr, enc, mlp, c2w, K


def test_render_view_equals_hand_loop():
    from human_body_reconstruction_b200 import ops
    g, vr, enc, mlp, c2w, K = _view_setup()
    H, W = vr.H, vr.W
    V = c2w.shape[0]
    for amp in (None, torch.bfloat16):
        with torch.autocast("cuda", dtype=amp or torch.bfloat16, enabled=amp is not None):
            torch.manual_seed(9)
            rgb, depth, opacity = vr.render_view(mlp, c2w, 16, hierarchical=True, chunk=500)
            torch.manual_seed(9)
            parts = []
            with torch.no_grad():
                c = c2w.to(DEV)
                for first in range(0, V * H * W, 500):
                    n = min(500, V * H * W - first)
                    o, d, nrm, _ = ops.ray_gen(c, H, W, K, first=first, n_rays=n)
                    out = vr.render(mlp, d, o, 16, dir_norm=nrm, hierarchical=True)
                    parts.append((out.rgb_fine, out.depth_fine, out.opacity_fine))
        assert rgb.shape == (V, H, W, 3) and depth.shape == (V, H, W) and opacity.shape == (V, H, W)
        assert torch.equal(rgb.reshape(-1, 3), torch.cat([p[0] for p in parts]))
        assert torch.equal(depth.reshape(-1), torch.cat([p[1] for p in parts]))
        assert torch.equal(opacity.reshape(-1), torch.cat([p[2] for p in parts]))


def test_render_view_matches_oracle_and_not_the_chunk():
    """2 views of 24 x 32 with fixed t against port.get_od + the oracle's vol_render (maps from its weights).  The device
    ray generator agrees with get_od to ~1 ulp, which the finest hash levels amplify, hence 1e-4 norm-wise.  With t given
    nothing is drawn, so the result is bit-identical for any chunk size."""
    g, vr, enc, mlp, c2w, K = _view_setup()
    H, W, V = vr.H, vr.W, c2w.shape[0]
    t = port.strat_t(g["near"], g["far"], 24, g["coarse__u_t"])
    res = [vr.render_view(mlp, c2w, 24, hierarchical=False, chunk=c, t=t.to(DEV)) for c in (97, 500, 1 << 16)]
    for r in res[1:]:
        assert all(torch.equal(a, b) for a, b in zip(res[0], r))
    rgb, depth, opacity = res[0]
    o, d, n = port.get_od(H, W, K, c2w)
    o, d, n = o.reshape(-1, 3), d.reshape(-1, 3), n.reshape(-1, 1)
    C, w, D, A = _oracle_maps(mlp_params(g, "mlp__"), g["tables"], g, t, n, o, d)
    Cr, _, _ = port.vol_render(mlp_params(g, "mlp__"), g["tables"], g["mu"], g["sigma"], g["scales"], d, o, t, n)
    assert torch.equal(C, Cr)
    assert rel(rgb.reshape(-1, 3), C) < 1e-4 and rel(depth.reshape(-1), D) < 1e-4 and rel(opacity.reshape(-1), A) < 1e-4


def test_render_view_memory_is_bounded_by_the_chunk_and_no_gradient_buffers():
    """Peak memory grows with the image only by the output maps (20 B per pixel), not by the rays or samples; under no_grad
    no table gradient buffer is allocated or zeroed (fp32 route through HashEncoder.forward, autocast route through the
    chained field node)."""
    g, vr, enc, mlp, c2w, K = _view_setup(H=48, W=64)
    t = port.strat_t(g["near"], g["far"], 24, g["coarse__u_t"]).to(DEV)

    def boom():
        raise AssertionError("a table gradient buffer was allocated under no_grad")

    enc._zeroed_grad_async = boom
    peaks = []
    for H, W in ((48, 64), (192, 256)):
        vr.H, vr.W = H, W
        for amp in (None, torch.bfloat16):
            with torch.autocast("cuda", dtype=amp or torch.bfloat16, enabled=amp is not None):
                vr.render_view(mlp, c2w, 24, hierarchical=True, chunk=256, t=t)        # warm-up of every shape
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                out = vr.render_view(mlp, c2w, 24, hierarchical=True, chunk=256, t=t)
                torch.cuda.synchronize()
                peaks.append(torch.cuda.max_memory_allocated() - base)
                del out
    grow = 2 * (192 * 256 - 48 * 64) * 20                                # 2 views x output bytes
    for small, big in zip(peaks[:2], peaks[2:]):
        assert big - small <= grow + (1 << 20), (small, big, grow)
