"""SURVEY 8f row 4: on-disk formats.  The scene readers are checked against fixtures produced by the reference's own
dataset classes (oracle/make_golden.py: gold_formats -> tests/golden/formats.npz over the two tiny scenes committed under
tests/golden/scene_*); bounds / density grid / checkpoints against the reference's literal save / load statements."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, load_golden, mlp_params
from human_body_reconstruction_b200 import formats


@pytest.mark.parametrize("flavour", ["blender", "new"])
def test_scene_readers_match_reference_datasets(flavour):
    g = load_golden("formats.npz")
    jpath = os.path.join(GOLDEN, "scene_" + flavour, "transforms_train.json")
    meta = formats.read_transforms(jpath)
    pre = flavour + "__"
    assert meta["flavour"] == flavour
    assert int(meta["H"]) == int(g[pre + "H"]) and int(meta["W"]) == int(g[pre + "W"])
    for k in ("focal1", "focal2", "cx", "cy"):
        assert float(meta[k]) == pytest.approx(float(g[pre + k]), rel=0, abs=0), k       # same float32 / python-float value
    assert torch.equal(meta["c2w"], g[pre + "c2w"])
    assert np.array_equal(np.array(meta["extra"], dtype=np.float64), g[pre + "extra"].numpy())
    K = formats.intrinsics_matrix(meta)
    assert K.dtype == torch.int64 and torch.equal(K, g[pre + "K"])                       # truncated like train_hash2.py:67-72
    images, c2w, K2, _ = formats.load_scene(jpath)
    assert images.dtype == torch.uint8 and images.shape == (2, int(g[pre + "H"]), int(g[pre + "W"]), 3)
    # torchvision's ToTensor of the reference == uint8 / 255, channel first
    assert torch.equal(images.permute(0, 3, 1, 2).float() / 255, g[pre + "images"])
    assert torch.equal(c2w, g[pre + "c2w"]) and torch.equal(K2, K)


def test_missing_files_raise():
    with pytest.raises(FileNotFoundError):
        formats.read_transforms("/nonexistent/transforms.json")
    with pytest.raises(FileNotFoundError):
        formats.read_image_u8("/nonexistent/x.png")


def test_bounds_round_trip_and_reference_statements(tmp_path):
    mn, mx = torch.tensor([-4.27, -4.31, -3.95]), torch.tensor([4.28, 4.27, 2.37])
    p = str(tmp_path / "bounds_model.npy")
    formats.save_bounds(p, mn, mx)
    want = torch.stack([mn, mx]).numpy()                                    # train_hash2.py:115
    assert np.array_equal(np.load(p), want) and np.load(p).dtype == np.float32
    bounds = np.load(p)                                                     # nerf2mesh.py:27-28
    lo, hi = formats.load_bounds(p)
    assert np.array_equal(lo, bounds[0]) and np.array_equal(hi, bounds[1])
    np.save(p, np.zeros((3, 3)))
    with pytest.raises(ValueError):
        formats.load_bounds(p)


def test_density_grid_layout(tmp_path):
    res = 4
    mn, mx = np.array([0.0, 10.0, 20.0]), np.array([1.0, 11.0, 21.0])
    x, y, z = (np.linspace(mn[i], mx[i], res) for i in range(3))
    X, Y, Z = np.meshgrid(x, y, z)                                          # nerf2mesh.py:30-37 ('xy' indexing)
    flat = np.stack([X.reshape(-1), Y.reshape(-1), Z.reshape(-1), X.reshape(-1) + Y.reshape(-1)], axis=1).astype(np.float32)
    grid = flat.reshape(res, res, res, 4)                                   # nerf2mesh.py:86
    p = str(tmp_path / "density_grid_w_rgb.npy")
    formats.save_density_grid(p, torch.from_numpy(grid))
    out, density = formats.load_density_grid(p)
    assert torch.equal(out, torch.from_numpy(grid)) and torch.equal(density, out[..., -1])
    a0, a1, a2 = formats.grid_axes(mn, mx, res)                             # axis 0 = y, axis 1 = x, axis 2 = z
    i, j, k = 2, 1, 3
    assert out[i, j, k, 0] == np.float32(a1[j]) and out[i, j, k, 1] == np.float32(a0[i]) and out[i, j, k, 2] == np.float32(a2[k])
    with pytest.raises(ValueError):
        formats.save_density_grid(p, np.zeros((4, 4, 3, 4)))


def test_checkpoint_names_and_dataparallel_prefix(tmp_path):
    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.sig_model = torch.nn.Sequential(torch.nn.Linear(3, 2))

    torch.manual_seed(0)
    net, enc = torch.nn.DataParallel(Net()), torch.nn.Embedding(4, 2)
    name = str(tmp_path / "run")
    formats.save_checkpoint(name, net, enc)
    n_path, e_path = formats.checkpoint_paths(name)
    assert n_path.endswith("run_Nerf_hash.pth") and e_path.endswith("run_encoder_hash.pth")
    assert list(torch.load(n_path).keys())[0] == "module.sig_model.0.weight"      # the reference's key (train_hash2.py:127,299)
    bare, enc2 = Net(), torch.nn.Embedding(4, 2)
    formats.load_checkpoint(name, bare, enc2)                                     # prefix stripped for an unwrapped module
    # nn.DataParallel moves its module to cuda:0 where there is a GPU: the weights are compared on the host
    assert torch.equal(bare.sig_model[0].weight, net.module.sig_model[0].weight.cpu()) and torch.equal(enc2.weight, enc.weight)
    torch.save(bare.state_dict(), n_path)
    wrapped = torch.nn.DataParallel(Net())
    formats.load_checkpoint(name, wrapped, enc2)                                  # and added for a wrapped one
    assert torch.equal(wrapped.module.sig_model[0].weight.cpu(), bare.sig_model[0].weight)


def test_checkpoint_keys_and_shapes_match_the_reference_classes(tmp_path):
    """What train_hash2.py:299-300 saves from the drop-in classes has the keys and shapes of the reference's own: its
    MLP_3D state_dict (tests/golden/mlp.npz, written by the unmodified reference) behind nn.DataParallel's prefix, and one
    (T, F) table per level of its HashEncoder.Embedding_list (tests/golden/hash_pow2.npz: L=16, T=1024, F=2)."""
    import human_body_reconstruction_b200 as hbr
    L, T, F = load_golden("hash_pow2.npz")["tables"].shape
    enc = hbr.HashEncoder(N_min=16, N_max=2048.0, L=L, F=F, T=T, dim=3, mu=torch.zeros(3), sigma=torch.tensor(1.0))
    mlp = hbr.MLP_3D(num_sig=2, num_col=2, L=L, F=F, d_view=24, max_bound=torch.ones(3), min_bound=-torch.ones(3))
    name = str(tmp_path / "m")
    formats.save_checkpoint(name, torch.nn.DataParallel(mlp), enc)
    n_path, e_path = formats.checkpoint_paths(name)
    nerf, encd = torch.load(n_path, map_location="cpu"), torch.load(e_path, map_location="cpu")
    ref_mlp = mlp_params(load_golden("mlp.npz"))
    assert {k: tuple(v.shape) for k, v in nerf.items()} == {"module." + k: tuple(v.shape) for k, v in ref_mlp.items()}
    assert {k: tuple(v.shape) for k, v in encd.items()} == {f"Embedding_list.{i}.weight": (T, F) for i in range(L)}
