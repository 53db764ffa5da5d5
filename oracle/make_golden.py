"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by executing the UNMODIFIED reference
(CPU, through oracle/ref_loader.py: the copy build() staged in oracle/_ref, or the checkout HBR_REFERENCE_DIR names):

    python oracle/make_golden.py

The fixtures hold explicit inputs and the reference's outputs, so consumers need neither the
reference tree nor a matching RNG.  Everything is float32/int64 unless noted.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
MU = torch.tensor([-4.27, -4.31, -3.95])
MAXB = torch.tensor([4.28, 4.27, 2.37])
SIGMA = ((MAXB - MU) ** 2).sum().sqrt()          # train_hash2.py:119


def npz(name, **kw):
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name), **{k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v))
                                                    for k, v in kw.items()})
    print("wrote", name, {k: tuple(np.asarray(v.detach() if torch.is_tensor(v) else v).shape) for k, v in kw.items()})


def build(ref, L, T, n_max, seed, table_scale):
    torch.manual_seed(seed)
    with ref_loader.quiet():
        enc = ref.hash_encoding.HashEncoder(N_min=16, N_max=n_max, L=L, F=2, T=T, dim=3, mu=MU, sigma=SIGMA, device="cpu")
        mlp = ref.test_hash.MLP_3D(num_sig=2, num_col=2, L=L, F=2, d_view=24, max_bound=ref.Bound(MAXB), min_bound=ref.Bound(MU))
        pe = ref.encoder.PositionalEncoder(3, 4)
    pe.sinus_in = pe.sinus_in.cpu()
    with torch.no_grad():
        for e in enc.Embedding_list:
            e.weight.mul_(table_scale)           # "trained-like" magnitudes; init is U(-1e-4,1e-4) (hash_encoding.py:32)
    return enc, mlp, pe


def points(n, seed):
    g = torch.Generator().manual_seed(seed)
    x = MU + torch.rand(n, 3, generator=g) * (MAXB - MU)
    x[:8] = MU - torch.rand(8, 3, generator=g)              # outside the bbox: negative cells / negative frac (Q4)
    x[8] = MU                                               # exactly on the corner
    x[9] = MAXB
    return x


def gold_hash(ref):
    for tag, L, T in (("pow2", 16, 1024), ("npow2", 4, 1000)):
        enc, _, _ = build(ref, L, T, 2048.0, 11, 1e4)
        x = points(257, 3)
        tables = torch.stack([e.weight.detach().clone() for e in enc.Embedding_list])
        scales = torch.stack([(enc.N_min * enc.b ** i).float() for i in range(L)])
        idx = []
        for i in range(L):                                   # hash_encoding.py:153-162, index part only
            un_x = ((x - enc.mu) / enc.sigma) * scales[i]
            x_val = torch.stack([un_x.long(), un_x.long() + 1], dim=-1)[..., None, :, :]
            bm = enc.bin_mask.reshape((1,) + (8, 3))
            idx.append(enc.hash_func(torch.where(bm, x_val[..., 0], x_val[..., 1]), T))
        with ref_loader.quiet():
            y = enc(x)
            y16 = enc(x.half())
        dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(4))
        y.backward(dy)
        g = torch.stack([e.weight.grad for e in enc.Embedding_list])
        npz(f"hash_{tag}.npz", x=x, tables=tables, mu=MU, sigma=SIGMA, scales=scales, n_min=16, n_max=2048.0,
            idx=torch.stack(idx), y=y.detach(), y_from_f16=y16.detach(), dy=dy, dtables=g)


def gold_mlp_dir(ref):
    _, mlp, pe = build(ref, 16, 64, 2048.0, 12, 1.0)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        mlp.sig_model[4].bias[0] += 1.0                      # so LeakyReLU sees both signs
    d = torch.nn.functional.normalize(torch.randn(96, 3, generator=g), dim=-1)
    enc_d = pe(d).reshape(96, -1)
    enc_d16 = pe(d.half()).reshape(96, -1)
    npz("dir.npz", d=d, enc=enc_d, enc_from_f16=enc_d16.float())
    feat = torch.randn(96, 32, generator=g).requires_grad_()
    dirs = enc_d.clone().requires_grad_()
    with ref_loader.quiet():
        out = mlp(feat, dirs)
        dens = mlp(feat)
    dout = torch.randn(out.shape, generator=g)
    out.backward(dout)
    kw = {k.replace(".", "__"): v.detach() for k, v in mlp.state_dict().items()}
    kw.update({"grad__" + k.replace(".", "__"): v.grad for k, v in mlp.named_parameters()})
    npz("mlp.npz", feat=feat.detach(), dirs=dirs.detach(), out=out.detach(), density_only=dens.detach(), dout=dout,
        dfeat=feat.grad, ddirs=dirs.grad, **kw)


def gold_mlp_autocast(ref):
    """The reference's own MLP_3D under torch.autocast (train_hash2.py:218 runs float16) against itself in fp32, on the
    CPU: the reference's 16-bit gradients differ from its fp32 ones by percents (ReLU-mask flips at pre-activations
    near zero), which is the yardstick the tensor-core kernels are held to (tests/test_gpu_precision.py)."""
    _, mlp, pe = build(ref, 16, 64, 2048.0, 12, 1.0)
    g = torch.Generator().manual_seed(15)
    R, S = 8, 128
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    dirs = pe(d).reshape(R, -1)
    feat = torch.randn(R * S, 32, generator=g) * 0.5
    dout = torch.randn(R * S, 4, generator=g)
    drep = dirs[:, None, :].repeat(1, S, 1).reshape(R * S, -1)          # vol_renderer.py:177-183
    kw = {k.replace(".", "__"): v.detach().clone() for k, v in mlp.state_dict().items()}
    for tag, dt in (("f32", None), ("f16", torch.float16), ("bf16", torch.bfloat16)):
        f = feat.clone().requires_grad_()
        for p_ in mlp.parameters():
            p_.grad = None
        with ref_loader.quiet(), torch.autocast("cpu", dtype=dt, enabled=dt is not None):
            out = mlp(f, drep)
        out.float().backward(dout)
        kw[f"{tag}__out"] = out.detach().float()
        kw[f"{tag}__dfeat"] = f.grad.clone()
        for k, v in mlp.named_parameters():
            kw[f"{tag}__grad__" + k.replace(".", "__")] = v.grad.clone()
    npz("mlp_autocast.npz", feat=feat, dirs=dirs, dout=dout, S=S, **kw)


def gold_composite(ref):
    g = torch.Generator().manual_seed(6)
    R, S = 48, 40
    t = torch.linspace(2.0, 6.0, S) + torch.rand(S, generator=g) * 4.0 / S
    rgb = torch.randn(R, S, 3, generator=g).requires_grad_()
    sig = (torch.randn(R, S, generator=g) * 6)
    sig[0, :6] = -25.0                                       # exercises the -10 clamp (helper.py:76)
    sig[1] = sig[1].abs() * 20                               # saturating ray: T underflows
    sig = sig.requires_grad_()
    dn = 1 + torch.rand(R, 1, generator=g)
    C, w, _ = ref.helper.calc_color(t=t, rgb=rgb, sigma=sig * 1.0, dir_norm=dn, device="cpu")
    gC = torch.randn(R, 3, generator=g)
    C.backward(gC)
    npz("composite.npz", t=t, rgb=rgb.detach(), sigma=sig.detach(), dir_norm=dn, C=C.detach(), w=w.detach()[..., 0],
        gC=gC, drgb=rgb.grad, dsigma=sig.grad)
    # per-ray depths (the fine pass hands calc_color an (R,2S) t)
    t2 = torch.sort(2 + 4 * torch.rand(R, S, generator=g), dim=-1).values
    rgb2 = torch.randn(R, S, 3, generator=g).requires_grad_()
    sig2 = (torch.randn(R, S, generator=g) * 6).requires_grad_()
    C2, w2, _ = ref.helper.calc_color(t=t2, rgb=rgb2, sigma=sig2 * 1.0, dir_norm=dn, device="cpu")
    C2.backward(gC)
    npz("composite_perray.npz", t=t2, rgb=rgb2.detach(), sigma=sig2.detach(), dir_norm=dn, C=C2.detach(),
        w=w2.detach()[..., 0], gC=gC, drgb=rgb2.grad, dsigma=sig2.grad)
    # hierarchical sampling (helper.py:23-51): replay the two torch.rand draws
    ro = torch.randn(R, 3, generator=g)
    rd = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
    near, far = torch.tensor(2.0), torch.tensor(6.0)
    torch.manual_seed(21)
    with ref_loader.quiet():
        rays_f, t_f = ref.helper.hierarchical_sampling(ro, rd, z_vals=t, weights=w.detach().clone(), n_samples=S,
                                                       tn=near, tf=far, device="cpu")
    torch.manual_seed(21)
    u_rs = torch.rand(R, S)
    u_s = torch.rand(S)
    npz("hier.npz", w=w.detach()[..., 0], t=t, near=2.0, far=6.0, u_rs=u_rs, u_s=u_s, rays_o=ro, rays_d=rd,
        t_fine=t_f, rays_fine=rays_f)


def gold_volrender(ref):
    """Full vol_render + loss + backward.  ReLU / LeakyReLU kinks make the gradient discontinuous in the
    pre-activations: a fixture with a pre-activation within rounding distance of 0 would pin an arbitrary mask
    choice, not arithmetic.  Seeds are therefore scanned until every pre-activation of both passes is at least
    2e-6 away from 0 (GPU/CPU pre-activations differ by ~3e-8), which makes the 1e-5 gradient tolerance of the GPU tests well-posed."""
    L, T, S, R = 16, 1024, 24, 40
    near, far = torch.tensor(2.0), torch.tensor(6.0)
    for seed in range(39, 400):
        enc, mlp, pe = build(ref, L, T, 2048.0, seed, 3e3)
        with torch.no_grad():
            mlp.sig_model[4].bias[0] += 1.5
        margin = [1e9]

        def hook(_m, _i, out, margin=margin, idx=None):
            margin[0] = min(margin[0], float(out.detach().abs().min()))
        hs = [m.register_forward_hook(hook) for m in (mlp.sig_model[0], mlp.sig_model[2], mlp.col_model[0], mlp.col_model[2])]
        hs.append(mlp.sig_model[4].register_forward_hook(lambda _m, _i, out: margin.__setitem__(0, min(margin[0], float(out.detach()[:, 0].abs().min())))))
        vr = ref.vol_renderer.Volume_Renderer(H=8, W=8, K=torch.eye(3), near=near, far=far, device="cpu", Pos_encode=enc,
                                              Dir_encode=pe, max_dim=64, sigma_val=SIGMA, mu=MU)
        g = torch.Generator().manual_seed(8)
        ro = torch.tensor([[0.5, -0.3, 4.0]]).repeat(R, 1) + 0.05 * torch.randn(R, 3, generator=g)
        rd = torch.nn.functional.normalize(-ro + 0.6 * torch.randn(R, 3, generator=g), dim=-1)
        dn = 1 + 0.2 * torch.rand(R, 1, generator=g)
        gt = torch.rand(R, 3, generator=g)
        kw = dict(rays_o=ro, rays_d=rd, dir_norm=dn, gt=gt, mu=MU, sigma=SIGMA, near=2.0, far=6.0, seed=seed,
                  tables=torch.stack([e.weight.detach().clone() for e in enc.Embedding_list]),
                  scales=torch.stack([(enc.N_min * enc.b ** i).float() for i in range(L)]))
        kw.update({"mlp__" + k.replace(".", "__"): v.detach().clone() for k, v in mlp.state_dict().items()})
        for hier in (False, True):
            tag = "hier" if hier else "coarse"
            for prm in list(enc.parameters()) + list(mlp.parameters()):
                prm.grad = None
            torch.manual_seed(31)
            with ref_loader.quiet():
                Cr, Cf, _ = vr.vol_render(mlp, rd, ro, num_samples=S, update_mask=False, dir_norm=dn, hierarchical=hier)
            loss = torch.nn.functional.mse_loss(Cr, gt) + torch.nn.functional.mse_loss(Cf, gt)   # train_hash2.py:221,177
            loss.backward()
            torch.manual_seed(31)
            kw[f"{tag}__u_t"] = torch.rand(S)
            if hier:
                kw[f"{tag}__u_rs"] = torch.rand(R, S)
                kw[f"{tag}__u_s"] = torch.rand(S)
            kw[f"{tag}__Cr"] = Cr.detach()
            kw[f"{tag}__Cf"] = Cf.detach()
            kw[f"{tag}__loss"] = loss.detach()
            kw[f"{tag}__dtables"] = torch.stack([e.weight.grad for e in enc.Embedding_list])
            for k, v in mlp.named_parameters():
                kw[f"{tag}__grad__" + k.replace(".", "__")] = v.grad.clone()
        for h_ in hs:
            h_.remove()
        if margin[0] >= 2e-6:
            print("seed", seed, "min |pre-activation|", margin[0])
            kw["kink_margin"] = margin[0]
            npz("volrender.npz", **kw)
            return
    raise RuntimeError("no seed found")


def gold_grid(ref):
    """nerf2mesh.py:27-40,69-86 on a 12^3 grid (the script itself needs torchmcubes/open3d, absent here;
    the statements below are the same calls on the same objects)."""
    L, T, res = 16, 1024, 12
    enc, mlp, pe = build(ref, L, T, 2048.0, 14, 5e3)
    min_b, max_b = MU.numpy(), MAXB.numpy()
    x = np.linspace(min_b[0], max_b[0], res)
    y = np.linspace(min_b[1], max_b[1], res)
    z = np.linspace(min_b[2], max_b[2], res)
    X, Y, Z = np.meshgrid(x, y, z)
    grid = torch.stack([torch.tensor(X.reshape(-1)), torch.tensor(Y.reshape(-1)), torch.tensor(Z.reshape(-1))], dim=1).to(torch.float16)
    view = torch.zeros_like(grid, dtype=torch.float16)
    view[..., 2] = 1.0
    with torch.no_grad(), ref_loader.quiet():
        out = mlp(enc(grid), pe(view).reshape(view.shape[0], -1))
    kw = dict(min_bound=min_b, max_bound=max_b, res=res, grid_f16=grid.float(), out=out.reshape(res, res, res, 4),
              mu=MU, sigma=SIGMA, tables=torch.stack([e.weight.detach().clone() for e in enc.Embedding_list]),
              scales=torch.stack([(enc.N_min * enc.b ** i).float() for i in range(L)]))
    kw.update({"mlp__" + k.replace(".", "__"): v.detach().clone() for k, v in mlp.state_dict().items()})
    npz("grid.npz", **kw)


def gold_rays(ref):
    """get_od / find_bounding_box (helper.py:176-208,109-141) for a 3-camera 6x5 rig with int64 K (Q14)."""
    H, W = 5, 6
    K = torch.from_numpy(np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1]]))
    K[0, 0] = 7.9
    K[1, 1] = 7.9
    K[0, 2] = W / 2
    K[1, 2] = H / 2
    g = torch.Generator().manual_seed(9)
    c2w = torch.eye(4).repeat(3, 1, 1)
    q, _ = torch.linalg.qr(torch.randn(3, 3, 3, generator=g))
    c2w[:, :3, :3] = q
    c2w[:, :3, 3] = torch.randn(3, 3, generator=g) * 2
    o, d, n = ref.helper.get_od(H, W, K, c2w)
    loader = [(None, c2w[i:i + 2], None) for i in (0, 2)]
    with ref_loader.quiet():
        mx, mn = ref.helper.find_bounding_box(loader, near=torch.tensor(2.0), far=torch.tensor(6.0), K=K)
    npz("rays.npz", H=H, W=W, K=K, c2w=c2w, rays_o=o, rays_d=d, dir_norm=n, max_bound=mx, min_bound=mn)


def gold_sdf(ref):
    """SDF mode end to end (train_hash2.py:122-126,220-224 -> vol_renderer.py:165-223 -> helper.py:76-89 ->
    test_hash.py:59-60,78-105): Volume_Renderer(use_sdf=True, var_model=VarModel()), hierarchical=False (the fine pass of
    the reference passes no sample positions to calc_color and cannot run in SDF mode), loss = mse + mse + 0.1 * eikonal."""
    L, T, R, S = 16, 1024, 12, 16
    torch.manual_seed(21)
    with ref_loader.quiet():
        enc = ref.hash_encoding.HashEncoder(N_min=16, N_max=512.0, L=L, F=2, T=T, dim=3, mu=MU, sigma=SIGMA, device="cpu")
        mlp = ref.test_hash.MLP_3D(num_sig=2, num_col=2, L=L, F=2, d_view=24, use_sdf=True, max_bound=ref.Bound(MAXB),
                                   min_bound=ref.Bound(MU))
        pe = ref.encoder.PositionalEncoder(3, 4)
    pe.sinus_in = pe.sinus_in.cpu()
    with torch.no_grad():
        for e in enc.Embedding_list:
            e.weight.mul_(5e3)
    var = ref.helper.VarModel()
    with torch.no_grad():
        var.b.fill_(3.0)
    model = torch.nn.DataParallel(mlp)                      # helper.py:87 reaches through .module
    near, far = torch.tensor(2.0), torch.tensor(6.0)
    vr = ref.vol_renderer.Volume_Renderer(H=8, W=8, K=torch.eye(3), near=near, far=far, device="cpu", Pos_encode=enc,
                                          Dir_encode=pe, max_dim=64, sigma_val=SIGMA, mu=MU, use_sdf=True, var_model=var)
    g = torch.Generator().manual_seed(5)
    ro = torch.tensor([[0.5, -0.3, 4.0]]).repeat(R, 1) + 0.05 * torch.randn(R, 3, generator=g)
    rd = torch.nn.functional.normalize(-ro + 0.6 * torch.randn(R, 3, generator=g), dim=-1)
    dn = 1 + 0.2 * torch.rand(R, 1, generator=g)
    gt = torch.rand(R, 3, generator=g)
    t = torch.linspace(2.0, 6.0, S) + torch.rand(S, generator=g) * 4.0 / S
    with ref_loader.quiet():
        Cr, Cf, norm = vr.vol_render(model, rd, ro, num_samples=S, t=t, update_mask=False, dir_norm=dn, hierarchical=False)
        sdf_probe = mlp.forward_sdf(ref_pts := (ro[:, None, :] + rd[:, None, :] * t[None, :, None]).reshape(-1, 3), encoder=enc)
    loss = (torch.nn.functional.mse_loss(Cr, gt) + torch.nn.functional.mse_loss(Cf, gt)
            + 0.1 * ref.helper.eikonal_loss(norm))           # train_hash2.py:221-224
    loss.backward()
    kw = dict(rays_o=ro, rays_d=rd, dir_norm=dn, gt=gt, t=t, mu=MU, sigma=SIGMA, min_bound=MU, max_bound=MAXB, b=torch.tensor(3.0),
              tables=torch.stack([e.weight.detach().clone() for e in enc.Embedding_list]),
              scales=torch.stack([(enc.N_min * enc.b ** i).float() for i in range(L)]),
              Cr=Cr.detach(), norm=norm.detach(), sdf=sdf_probe.detach(), loss=loss.detach(), grad_b=var.b.grad.clone(),
              dtables=torch.stack([e.weight.grad for e in enc.Embedding_list]))
    kw.update({"mlp__" + k.replace(".", "__"): v.detach().clone() for k, v in mlp.state_dict().items()})
    for k, v in mlp.named_parameters():
        kw["grad__" + k.replace(".", "__")] = v.grad.clone()
    npz("sdf.npz", **kw)


def gold_formats():
    """dataset.py / dataset_new.py readers of the reference on two tiny scenes written here (tests/golden/scene_*), plus
    the int64 K the trainer builds from them (train_hash2.py:67-72)."""
    import importlib
    import json
    import cv2
    rng = np.random.default_rng(4)
    H, W, V = 5, 6, 2
    kw = {}
    for flavour in ("blender", "new"):
        root = os.path.join(OUT, "scene_" + flavour)
        os.makedirs(os.path.join(root, "train"), exist_ok=True)
        frames = []
        for v in range(V):
            img = rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
            name = f"r_{v}"
            cv2.imwrite(os.path.join(root, "train", name + ".png"), img)          # cv2 writes BGR
            m = np.eye(4)
            m[:3, :4] = rng.normal(size=(3, 4))
            fr = {"file_path": f"./train/{name}" + (".png" if flavour == "new" else ""), "transform_matrix": m.tolist()}
            fr["sharpness" if flavour == "new" else "rotation"] = float(rng.uniform())
            frames.append(fr)
        meta = {"camera_angle_x": 0.6911112070083618, "frames": frames}
        if flavour == "new":
            meta.update(w=W, h=H, fl_x=7.9, fl_y=8.2, cx=3.4, cy=2.6)
        jpath = os.path.join(root, "transforms_train.json")
        with open(jpath, "w") as f:
            json.dump(meta, f)
        sys.path.insert(0, ref_loader.REF_DIR)
        try:
            mod = importlib.import_module("dataset_new" if flavour == "new" else "dataset")
        finally:
            sys.path.remove(ref_loader.REF_DIR)
        ds = (mod.NeRF_DATA_NEW if flavour == "new" else mod.NeRF_DATA)(json_path=jpath)
        items = [ds[i] for i in range(len(ds))]
        K = torch.from_numpy(np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1]]))               # train_hash2.py:67-72
        K[0, 0] = ds.focal1
        K[1, 1] = ds.focal2
        K[0, 2] = ds.cx
        K[1, 2] = ds.cy
        pre = flavour + "__"
        kw.update({pre + "H": int(ds.H), pre + "W": int(ds.W), pre + "focal1": float(ds.focal1), pre + "focal2": float(ds.focal2),
                   pre + "cx": float(ds.cx), pre + "cy": float(ds.cy), pre + "K": K,
                   pre + "images": torch.stack([it[0] for it in items]), pre + "c2w": torch.stack([it[1] for it in items]),
                   pre + "extra": np.array([it[2] for it in items], dtype=np.float64)})
        for m in ("dataset", "dataset_new"):
            sys.modules.pop(m, None)
    npz("formats.npz", **kw)


if __name__ == "__main__":
    ref = ref_loader.load()
    gold_hash(ref)
    gold_mlp_dir(ref)
    gold_mlp_autocast(ref)
    gold_composite(ref)
    gold_volrender(ref)
    gold_grid(ref)
    gold_rays(ref)
    gold_sdf(ref)
    gold_formats()
