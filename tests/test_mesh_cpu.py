"""CPU: the float64 position-gradient oracle (tests/mesh_oracle.py) against central differences, the index -> world map of
mesh.extract_mesh against the coordinates the density grid is evaluated at, and the binary PLY round trip."""
import os

import numpy as np
import pytest
import torch

import mesh_oracle
from oracle import port

from human_body_reconstruction_b200 import formats, mesh


def _field(T=2 ** 12, L=16, F=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    tables = (torch.rand(L, T, F, generator=g, dtype=torch.float64) * 2 - 1)
    scales = port.level_scales(16, 2048.0, L)
    return tables, scales


@pytest.mark.parametrize("T", [2 ** 12, 3001])
def test_oracle_dx_matches_central_differences(T):
    tables, scales = _field(T)
    mu, sigma = [-1.0, -1.2, -0.9], 3.4
    g = torch.Generator().manual_seed(1)
    x = torch.rand(400, 3, generator=g, dtype=torch.float64) * 1.8 - 0.9
    dy = torch.randn(400, 32, generator=g, dtype=torch.float64)
    h = 1e-7
    # keep the points whose +-h stencil stays inside one cell on every level (the encoding is trilinear there: linear
    # along each axis, so central differences are exact up to rounding)
    mu64 = torch.tensor(mu, dtype=torch.float64)
    ok = torch.ones(x.shape[0], dtype=torch.bool)
    for s in scales.tolist():
        c0 = (((x - mu64) / sigma) * s).trunc()
        for a in range(3):
            for sgn in (-1, 1):
                xs = x.clone()
                xs[:, a] += sgn * h
                ok &= ((((xs - mu64) / sigma) * s).trunc() == c0).all(1)
    assert ok.sum() > 300
    x, dy = x[ok], dy[ok]
    ana = mesh_oracle.hash_dx64(x, tables, mu, sigma, scales, dy, frac_from_fp32=False)
    fd = torch.empty_like(ana)
    for a in range(3):
        xp, xm = x.clone(), x.clone()
        xp[:, a] += h
        xm[:, a] -= h
        yp = mesh_oracle.encode64(xp, tables, mu, sigma, scales, frac_from_fp32=False)
        ym = mesh_oracle.encode64(xm, tables, mu, sigma, scales, frac_from_fp32=False)
        fd[:, a] = ((yp - ym) * dy).sum(1) / (2 * h)
    err = float((ana - fd).norm() / ana.norm())
    print(f"T={T}: oracle dx vs central differences {err:.2e} over {x.shape[0]} points")
    assert err < 1e-7


def test_index_to_world_matches_grid_points():
    mn, mx, res = [-1.3, -0.7, -2.1], [1.1, 0.9, 0.4], 37
    axes = mesh.world_axes(mn, mx, res)
    pts = port.grid_points(np.array(mn), np.array(mx), res).float()          # flat p = (i*res + j)*res + k <-> (x[j], y[i], z[k])
    y, x, z = formats.grid_axes(mn, mx, res)
    X, Y, Z = np.meshgrid(x, y, z)
    ref = torch.from_numpy(np.stack([X, Y, Z], axis=-1).astype(np.float16).astype(np.float32)).reshape(-1, 3)
    assert torch.equal(pts, ref)
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, res, (2000, 3), generator=g)
    idx[0] = torch.tensor([res - 1] * 3)
    idx[1] = 0
    w = mesh.index_to_world(idx.float(), axes)
    p = (idx[:, 0] * res + idx[:, 1]) * res + idx[:, 2]
    assert torch.equal(w, ref[p])
    # linear between grid points, along each index axis separately (marching-cubes vertices lie on grid edges)
    for a in range(3):
        lo = torch.randint(0, res - 1, (500, 3), generator=g)
        t = torch.rand(500, generator=g)
        v = lo.float()
        v[:, a] += t
        hi = lo.clone()
        hi[:, a] += 1
        wl, wh = mesh.index_to_world(lo.float(), axes), mesh.index_to_world(hi.float(), axes)
        want = wl + t[:, None] * (wh - wl)
        assert torch.allclose(mesh.index_to_world(v, axes), want, rtol=0, atol=1e-6)
    # the end point: an index of exactly res - 1 along an axis maps to the last coordinate
    e = mesh.index_to_world(torch.tensor([[res - 1.0, 0.0, 0.0]]), axes)
    assert float(e[0, 1]) == float(np.float16(mx[1]))


def _mesh(nv=1000, nf=1900, seed=0):
    g = torch.Generator().manual_seed(seed)
    n = torch.randn(nv, 3, generator=g)
    c = torch.rand(nv, 3, generator=g) * 1.4 - 0.2                          # raw colours: some outside [0, 1]
    c[0] = torch.tensor([float("nan"), 1.0, 0.0])
    return mesh.Mesh(torch.randn(nv, 3, generator=g), torch.randint(0, nv, (nf, 3), generator=g, dtype=torch.int32),
                     n / n.norm(dim=1, keepdim=True), c)


def test_write_read_ply_round_trip(tmp_path):
    m = _mesh()
    path = os.path.join(tmp_path, "m.ply")
    mesh.write_ply(path, m)
    head = open(path, "rb").read().split(b"end_header\n")[0].decode().splitlines()
    assert head[:2] == ["ply", "format binary_little_endian 1.0"]
    assert "element vertex 1000" in head and "element face 1900" in head
    assert head[-1] == "property list uchar int vertex_indices"
    assert os.path.getsize(path) == len("\n".join(head)) + len("\nend_header\n") + 1000 * 27 + 1900 * 13
    r = mesh.read_ply(path)
    assert torch.equal(r.vertices, m.vertices) and torch.equal(r.normals, m.normals) and torch.equal(r.faces, m.faces)
    want = torch.round(torch.nan_to_num(m.colors, nan=0.0).clamp(0, 1) * 255).to(torch.uint8)
    assert r.colors.dtype == torch.uint8 and torch.equal(r.colors, want)
    assert int(r.colors[0, 0]) == 0 and int(r.colors[0, 1]) == 255


def test_ply_empty_mesh_and_bad_header(tmp_path):
    path = os.path.join(tmp_path, "e.ply")
    e = mesh.Mesh(torch.zeros(0, 3), torch.zeros(0, 3, dtype=torch.int32), torch.zeros(0, 3), torch.zeros(0, 3))
    mesh.write_ply(path, e)
    r = mesh.read_ply(path)
    assert r.vertices.shape == (0, 3) and r.faces.shape == (0, 3)
    with open(path, "r+b") as f:
        f.write(b"plx")
    with pytest.raises(ValueError):
        mesh.read_ply(path)
