"""-m gpu: the sparse marching-cubes route (coarse lattice and brick densities, seed, closure, brick marching cubes, and
extract_mesh(sparse=True)) against the numpy restatement of the brick lattice in tests/sparse_mc_oracle.py and against the
dense route."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import sparse_mc_oracle as so
import test_sparse_mc_cpu as vols
from conftest import ROOT
from test_gpu_mesh import _ellipsoid, _field

pytestmark = pytest.mark.gpu
DEV = "cuda"


def hbr():
    import human_body_reconstruction_b200 as h
    return h


def cut_bricks(vol: torch.Tensor, bricks: torch.Tensor) -> torch.Tensor:
    """(n,9,9,9) values of the listed bricks of a dense (res,res,res) device tensor, indices clamped to res-1."""
    res = vol.shape[0]
    nb = so.brick_count(res)
    b = bricks.long()
    Bc = torch.stack((b // (nb * nb), (b // nb) % nb, b % nb), 1)
    ix = (8 * Bc[:, :, None] + torch.arange(9, device=vol.device)).clamp_(max=res - 1)         # (n,3,9)
    return vol[ix[:, 0, :, None, None], ix[:, 1, None, :, None], ix[:, 2, None, None, :]].contiguous()


def coarse_of(vol: torch.Tensor) -> torch.Tensor:
    ix = torch.from_numpy(so.lattice_index(vol.shape[0])).to(vol.device)
    return vol[ix[:, None, None], ix[None, :, None], ix[None, None, :]].contiguous()


def sparse_of(vol: torch.Tensor, iso: float):
    h = hbr()
    return h.mesh.sparse_surface_index(vol.shape[0], iso, coarse_of(vol), lambda b: cut_bricks(vol, b))


def active_of(surf, res):
    nb = so.brick_count(res)
    a = np.zeros(nb ** 3, dtype=bool)
    a[surf.bricks.cpu().numpy()] = True
    return a.reshape((nb,) * 3)


def ellipsoid_volume(res):
    h = hbr()
    q = h.mesh.world_axes([-1.0, -1.1, -0.9], [1.1, 0.9, 1.0], res, DEV).double()
    Yg, Xg, Zg = torch.meshgrid(q[0], q[1], q[2], indexing="ij")
    return _ellipsoid(Xg, Yg, Zg)[0].float().contiguous()


def synthetic(name, res):
    if name == "ellipsoid":
        return ellipsoid_volume(res), 0.0
    if name == "bumps":
        return torch.from_numpy(vols.smooth(res, 7)).to(DEV), 0.5
    return torch.from_numpy({"two_components": vols.two_components, "tube": vols.tube}[name](res)).to(DEV), 0.0


def check_against_oracle(vol, iso, surf):
    """Active set, rounds, vertex rows (bitwise) and face count against the oracle; faces index valid vertices."""
    v = vol.cpu().numpy()
    act, rounds = so.closure(v, iso)
    assert np.array_equal(active_of(surf, v.shape[0]), act) and surf.rounds == rounds
    bricks = surf.bricks.cpu().numpy()
    assert len(np.unique(bricks)) == len(bricks)
    got = surf.vertices.cpu().numpy()
    assert np.array_equal(so.sorted_rows(got), so.sorted_rows(so.crossing_vertices(v, iso, act)))
    assert surf.faces.shape[0] == so.triangle_count(v, iso, act)
    if surf.faces.shape[0]:
        assert int(surf.faces.min()) >= 0 and int(surf.faces.max()) < got.shape[0]
    assert surf.points == (so.brick_count(v.shape[0]) + 1) ** 3 + 729 * len(bricks)
    return act


def same_mesh_as_sets(va, fa, vb, fb):
    va, vb = np.asarray(va), np.asarray(vb)
    assert np.array_equal(so.sorted_rows(va), so.sorted_rows(vb))
    assert np.array_equal(so.face_triples(va, np.asarray(fa)), so.face_triples(vb, np.asarray(fb)))


@pytest.mark.parametrize("field", ["busy", "smooth"])
@pytest.mark.parametrize("res", [61, 64])
def test_coarse_and_brick_densities_equal_density_grid_bitwise(field, res):
    h = hbr()
    enc, mlp, _, mn, mx, _ = _field(coarse_only=field == "smooth")
    dense = h.mesh.density_grid(enc, mlp, None, mn, mx, res)
    table, geom, params, dims = h.mesh._native_field(enc, mlp)
    coarse = h.ops.coarse_density(mn, mx, res, table, geom, params, dims, chunk=5_000)
    assert torch.equal(coarse, coarse_of(dense))
    nb = so.brick_count(res)
    bricks = torch.arange(nb ** 3, device=DEV, dtype=torch.int32).flip(0)           # any order; the last bricks are clamped
    got = h.ops.brick_density(mn, mx, res, bricks, table, geom, params, dims, chunk=100_003)
    assert torch.equal(got, cut_bricks(dense, bricks))


@pytest.mark.parametrize("name,res", [("ellipsoid", 61), ("ellipsoid", 64), ("ellipsoid", 65), ("ellipsoid", 128),
                                      ("two_components", 64), ("tube", 65), ("bumps", 61), ("bumps", 128)])
def test_synthetic_volumes_match_the_oracle(name, res):
    h = hbr()
    vol, iso = synthetic(name, res)
    surf = sparse_of(vol, iso)
    act = check_against_oracle(vol, iso, surf)
    if name == "two_components":
        assert not act[4, 4, 4]                                     # the small ball is dropped
    if name == "tube":
        assert surf.rounds >= 7
    # every brick forced active: the dense marching cubes, vertex for vertex and face for face
    nb = so.brick_count(res)
    every = torch.arange(nb ** 3, device=DEV, dtype=torch.int32)
    bmap = every.view(nb, nb, nb).clone()
    vf, ff = h.ops.brick_mc(cut_bricks(vol, every), every, bmap, res, iso)
    vd, fd = h.mesh.marching_cubes(vol, iso)
    assert vf.shape[0] == vd.shape[0] and ff.shape[0] == fd.shape[0] > 0
    same_mesh_as_sets(vf.cpu(), ff.cpu(), vd.cpu(), fd.cpu())
    if so.covers_all_crossings(vol.cpu().numpy(), iso, act):
        same_mesh_as_sets(surf.vertices.cpu(), surf.faces.cpu(), vd.cpu(), fd.cpu())


def _iso(h, enc, mlp, mn, mx):
    return float(h.mesh.density_grid(enc, mlp, None, mn, mx, 64).float().median())


def _by_vertex(m):
    v = m.vertices.cpu().numpy()
    o = np.lexsort(v.T[::-1])
    return v[o], m.normals.cpu().numpy()[o], m.colors.cpu().numpy()[o]


@pytest.mark.parametrize("field,res", [("busy", 128), ("smooth", 128), ("busy", 256), ("smooth", 256), ("smooth", 512)])
def test_extract_mesh_sparse_on_the_test_fields(field, res):
    h = hbr()
    enc, mlp, denc, mn, mx, _ = _field(coarse_only=field == "smooth")
    iso = _iso(h, enc, mlp, mn, mx)
    dense = h.mesh.density_grid(enc, mlp, None, mn, mx, res)
    surf = h.mesh.sparse_field_surface(enc, mlp, mn, mx, res, iso)
    d = dense.cpu().numpy()
    del dense
    act = check_against_oracle(torch.from_numpy(d), iso, surf)
    covered = so.covers_all_crossings(d, iso, act)
    ms = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso, sparse=True)
    print(f"{field} res={res}: {act.sum()} of {act.size} bricks active in {surf.rounds} rounds, {ms.vertices.shape[0]} vertices, "
          f"covers every crossing cell: {covered}")
    assert ms.vertices.shape[0] == surf.vertices.shape[0] and ms.faces.shape[0] == surf.faces.shape[0]
    if covered:
        md = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso)
        same_mesh_as_sets(ms.vertices.cpu(), ms.faces.cpu(), md.vertices.cpu(), md.faces.cpu())
        vs, ns, cs = _by_vertex(ms)
        vd, nd, cd = _by_vertex(md)
        assert np.array_equal(vs, vd) and np.array_equal(ns, nd) and np.array_equal(cs, cd)
    else:
        assert ms.vertices.shape[0] == len(so.crossing_vertices(d, iso, act)) < so.port.mc_crossing_edges(d, iso)


def test_sparse_route_is_deterministic_and_handles_no_crossing():
    h = hbr()
    enc, mlp, denc, mn, mx, _ = _field()
    iso = _iso(h, enc, mlp, mn, mx)
    a = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=128, iso=iso, sparse=True)
    b = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=128, iso=iso, sparse=True)
    assert a.vertices.shape[0] > 0
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    empty = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=64, iso=1e30, sparse=True)
    assert empty.vertices.shape == (0, 3) and empty.faces.shape == (0, 3)
    assert empty.normals.shape == (0, 3) and empty.colors.shape == (0, 3)


def test_export_mesh_script_sparse(tmp_path):
    h = hbr()
    from human_body_reconstruction_b200 import formats
    work = str(tmp_path)
    enc, mlp, _, mn, mx, _ = _field(coarse_only=True)
    iso = _iso(h, enc, mlp, mn, mx)
    formats.save_checkpoint(os.path.join(work, "s"), torch.nn.DataParallel(mlp.cpu()), enc.cpu())
    formats.save_bounds(os.path.join(work, "bounds_model.npy"), torch.tensor(mn), torch.tensor(mx))
    out = os.path.join(work, "mesh.ply")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "export_mesh.py"), "--ckpt_name", "s", "--bound_pth",
                        "bounds_model.npy", "--hash_size", "14", "--res", "96", "--iso", repr(iso), "--sparse", "--out", out],
                       cwd=work, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    rep = json.loads(r.stdout.strip().splitlines()[-1])
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import export_mesh
    e2, n2, d2, lo, hi = export_mesh.build_field(os.path.join(work, "s"), os.path.join(work, "bounds_model.npy"), 14, 2048.0)
    m = h.mesh.extract_mesh(e2, n2, d2, lo, hi, res=96, iso=iso, sparse=True)
    back = h.mesh.read_ply(out)
    assert back.vertices.shape[0] == m.vertices.shape[0] == rep["vertices"] > 0
    assert back.faces.shape[0] == m.faces.shape[0] == rep["faces"] > 0
    assert rep["active_bricks"] > 0 and rep["rounds"] >= 1
    assert torch.equal(back.vertices, m.vertices.cpu()) and torch.equal(back.faces, m.faces.cpu())


def test_bounded_memory_at_2048_on_the_smooth_field():
    h = hbr()
    enc, mlp, _, mn, mx, _ = _field(coarse_only=True)
    iso = _iso(h, enc, mlp, mn, mx)
    res = 2048
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    surf = h.mesh.sparse_field_surface(enc, mlp, mn, mx, res, iso)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    n, nv, nf = surf.bricks.shape[0], surf.vertices.shape[0], surf.faces.shape[0]
    nb = so.brick_count(res)
    # the peak is the meshing stage: brick map, coarse lattice, per active brick its values (729 fp32), 16-bit edge ids
    # (3 x 729), slot and offsets, and the mesh; while the rounds are joined the values are held twice, without edge ids
    per_brick = max(2 * 729 * 4, 729 * 4 + 3 * 729 * 2) + 4 + 16
    bound = 4 * nb ** 3 + 4 * (nb + 1) ** 3 + n * per_brick + 12 * (nv + nf) + (1 << 19) * (6 + 128 + 4) + (64 << 20)
    print(f"2048^3 smooth field: {n} of {nb ** 3} bricks active ({n / nb ** 3:.4f}) in {surf.rounds} rounds, {nv} vertices, "
          f"{nf} faces; peak {peak / 1e9:.2f} GB, bound {bound / 1e9:.2f} GB, dense route {16 * res ** 3 / 1e9:.0f} GB")
    assert nv > 0 and peak <= bound and bound < 0.25 * 16 * res ** 3
