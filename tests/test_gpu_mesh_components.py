"""-m gpu: connected components of a triangle mesh (hbr_mesh_components, mesh.mesh_components) against the scipy oracle in
tests/mesh_cc_oracle.py on built graphs, marching-cubes meshes of synthetic volumes and the test fields; floater removal
(mesh.filter_components, extract_mesh's min_component_faces / largest_components, export_mesh.py's flags); dense against
sparse route after filtering; peak memory at 2048^3."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import mesh_cc_oracle as cc
import test_sparse_mc_cpu as vols
from conftest import ROOT
from test_gpu_mesh import _field
from test_gpu_mesh_sparse import _iso

pytestmark = pytest.mark.gpu
DEV = "cuda"


def hbr():
    import human_body_reconstruction_b200 as h
    return h


def check_against_oracle(faces, nv):
    """Labels and sizes bitwise against the oracle; returns the MeshComponents."""
    h = hbr()
    label, fc, vc = h.ops.mesh_components(faces, nv)
    o_label, o_fc, o_vc = cc.components(faces.cpu().numpy(), nv)
    assert label.dtype == fc.dtype == vc.dtype == torch.int32 and label.shape == (nv,)
    assert np.array_equal(label.cpu().numpy(), o_label)
    assert np.array_equal(fc.cpu().numpy(), o_fc) and np.array_equal(vc.cpu().numpy(), o_vc)
    comp = h.mesh.mesh_components(faces, nv)
    roots, sf, sv = cc.sizes(o_label, o_fc, o_vc)
    assert np.array_equal(comp.roots.cpu().numpy(), roots)
    assert np.array_equal(comp.faces.cpu().numpy(), sf) and np.array_equal(comp.vertices.cpu().numpy(), sv)
    return comp


# ---- built graphs ---------------------------------------------------------------------------------------------------
def random_components(sizes, isolated, seed):
    """Faces of len(sizes) connected pieces (a chain through each piece's vertices plus random faces inside it, degenerate
    ones included) and `isolated` unused vertices; vertex ids shuffled, face order and corner rotation shuffled."""
    rng = np.random.default_rng(seed)
    faces, base = [], 0
    for n in sizes:
        i = np.arange(n - 1)
        chain = np.stack((i, i + 1, rng.integers(0, n, n - 1)), 1)
        extra = rng.integers(0, n, (2 * n, 3))
        faces += [chain + base, extra + base]
        base += n
    nv = base + isolated
    f = np.concatenate(faces)
    f = np.take_along_axis(f, (np.arange(3)[None] + rng.integers(0, 3, (len(f), 1))) % 3, 1)
    f = rng.permutation(nv)[f][rng.permutation(len(f))]
    return torch.from_numpy(f.astype(np.int32)).to(DEV), nv


@pytest.mark.parametrize("sizes,isolated,seed", [([1000], 0, 0), ([3, 5, 2, 7], 4, 1), ([2] * 500 + [9000, 40000], 300, 2),
                                                 (list(range(2, 400)), 1000, 3)])
def test_random_meshes_with_known_components(sizes, isolated, seed):
    f, nv = random_components(sizes, isolated, seed)
    comp = check_against_oracle(f, nv)
    assert comp.roots.shape[0] == len(sizes) + isolated
    assert sorted(comp.vertices.tolist()) == sorted(list(sizes) + [1] * isolated)


def deep_path(n):
    """A path of n vertices whose faces (v, v-1, v-1) run from the highest id down."""
    v = torch.arange(n - 1, 0, -1, device=DEV, dtype=torch.int32)
    return torch.stack((v, v - 1, v - 1), 1).contiguous(), n


def star(n_faces, hub):
    """n_faces faces around one hub vertex (at the low end, the middle or the high end of the ids)."""
    nv = 2 * n_faces + 1
    h = {"low": 0, "mid": n_faces, "high": nv - 1}[hub]
    rim = torch.arange(nv, device=DEV, dtype=torch.int32)
    rim = rim[rim != h].view(-1, 2)
    return torch.cat((torch.full((n_faces, 1), h, device=DEV, dtype=torch.int32), rim), 1).contiguous(), nv


@pytest.mark.parametrize("case", ["path", "star_low", "star_mid", "star_high"])
def test_contention_cases_match_the_oracle_and_repeat_bitwise(case):
    h = hbr()
    f, nv = deep_path(1_000_001) if case == "path" else star(1_000_000, case.split("_")[1])
    comp = check_against_oracle(f, nv)
    assert comp.roots.tolist() == [0] and comp.faces.tolist() == [f.shape[0]] and comp.vertices.tolist() == [nv]
    a = h.ops.mesh_components(f, nv)
    b = h.ops.mesh_components(f, nv)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_no_faces_and_no_vertices():
    h = hbr()
    none = torch.zeros((0, 3), device=DEV, dtype=torch.int32)
    label, fc, vc = h.ops.mesh_components(none, 1000)
    assert torch.equal(label, torch.arange(1000, device=DEV, dtype=torch.int32))
    assert not fc.any() and bool((vc == 1).all())
    check_against_oracle(none, 1000)
    out = h.ops.mesh_components(none, 0)
    assert all(x.shape == (0,) for x in out)
    comp = h.mesh.mesh_components(none, 0)
    assert comp.roots.shape == (0,) and h.mesh.keep_components(comp, largest=1).shape == (0,)


# ---- marching-cubes meshes of synthetic volumes ----------------------------------------------------------------------
def mc_mesh(vol):
    h = hbr()
    return h.mesh.marching_cubes(torch.from_numpy(vol).to(DEV), 0.0)


def test_two_components_volume():
    v, f = mc_mesh(vols.two_components())
    comp = check_against_oracle(f, v.shape[0])
    assert comp.roots.shape[0] == 2 and int(comp.vertices.sum()) == v.shape[0] and int(comp.faces.sum()) == f.shape[0]


def test_balls_one_component_each_and_largest_keeps_the_biggest():
    h = hbr()
    centres, radii = [(12.0, 12.0, 12.0), (40.3, 14.2, 20.7), (22.5, 44.1, 43.6), (45.2, 46.8, 12.4)], [7.5, 4.2, 9.6, 2.3]
    vol = np.maximum.reduce([vols._ball(64, c, r) for c, r in zip(centres, radii)])
    v, f = mc_mesh(vol)
    comp = check_against_oracle(f, v.shape[0])
    assert comp.roots.shape[0] == 4
    m = h.mesh.Mesh(v, f, torch.zeros_like(v), torch.zeros_like(v))
    big = h.mesh.filter_components(m, largest=1)
    d = (big.vertices - torch.tensor(centres[2], device=DEV)).norm(dim=1)
    assert big.vertices.shape[0] == int(comp.vertices.max()) and bool((d - radii[2]).abs().max() < 1.0)
    two = h.mesh.filter_components(m, largest=2)
    assert two.faces.shape[0] == int(torch.topk(comp.faces, 2).values.sum())


def test_ball_inside_a_shell_gives_three_components():
    i, j, k = np.meshgrid(*(np.arange(64, dtype=np.float64),) * 3, indexing="ij")
    r = np.sqrt((i - 31.6) ** 2 + (j - 32.3) ** 2 + (k - 31.8) ** 2)
    vol = np.maximum(6.1 - r, np.minimum(r - 12.4, 20.7 - r)).astype(np.float32)
    v, f = mc_mesh(vol)
    comp = check_against_oracle(f, v.shape[0])
    assert comp.roots.shape[0] == 3
    # sizes grow with the sphere's radius: the ball's, the shell's inner wall, the shell's outer wall
    by_radius = [float(r) for r in (v - torch.tensor([31.6, 32.3, 31.8], device=DEV)).norm(dim=1)[comp.roots].tolist()]
    order = np.argsort(by_radius)
    assert list(comp.faces.cpu().numpy()[order]) == sorted(comp.faces.tolist())


# ---- the test fields -------------------------------------------------------------------------------------------------
def _sorted_rows(x):
    """rows of an (n, c) 32-bit tensor as int32 bit patterns, sorted lexicographically (stable sorts, last column first)."""
    x = x.contiguous().view(torch.int32)
    order = torch.arange(x.shape[0], device=x.device)
    for c in range(x.shape[1] - 1, -1, -1):
        order = order[torch.sort(x[order, c], stable=True).indices]
    return x[order]


def same_as_sets(a, b):
    """Vertex rows with their normals and colours as multisets, and faces as vertex triples up to rotation (winding kept)."""
    assert a.vertices.shape == b.vertices.shape and a.faces.shape == b.faces.shape
    ra, rb = (_sorted_rows(torch.cat((m.vertices, m.normals, m.colors), 1)) for m in (a, b))
    assert torch.equal(ra, rb)
    both = torch.cat((a.vertices, b.vertices)).contiguous().view(torch.int32)
    _, inv = torch.unique(both, dim=0, return_inverse=True)
    tri = []
    for m, ids in ((a, inv[:a.vertices.shape[0]]), (b, inv[a.vertices.shape[0]:])):
        r = ids[m.faces.long()]
        k = r.argmin(1, keepdim=True)
        tri.append(_sorted_rows(torch.gather(r, 1, (k + torch.arange(3, device=DEV)) % 3).to(torch.int32)))
    assert torch.equal(tri[0], tri[1])


FIELD_CASES = [(f, r) for r in (128, 256, 512) for f in ("busy", "smooth")]


@pytest.mark.parametrize("field,res", FIELD_CASES)
@pytest.mark.parametrize("sparse", [False, True], ids=["dense", "sparse"])
def test_filtering_the_test_fields(field, res, sparse):
    h = hbr()
    enc, mlp, denc, mn, mx, _ = _field(coarse_only=field == "smooth")
    iso = _iso(h, enc, mlp, mn, mx)
    m = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso, sparse=sparse)
    nv = m.vertices.shape[0]
    comp = check_against_oracle(m.faces, nv)
    top = int(comp.faces.max())
    print(f"{field} res={res} {'sparse' if sparse else 'dense'}: {nv} vertices, {comp.roots.shape[0]} components, the largest "
          f"{top} of {m.faces.shape[0]} faces")
    for kw in ({"min_faces": 64}, {"largest": 1}, {"min_faces": 16, "largest": 5}):
        f = h.mesh.filter_components(m, **kw)
        keep = h.mesh.keep_components(comp, **kw)
        assert f.faces.shape[0] == int(comp.faces[keep].sum()) > 0
        assert f.vertices.shape[0] == int(comp.vertices[keep].sum())
        # the kept vertices are rows of the unfiltered mesh, attributes and all, in their original order
        vi, _, _, _ = h.mesh.filter_by_components(m.vertices, m.faces, kw.get("min_faces", 0), kw.get("largest"))
        assert bool((vi[1:] > vi[:-1]).all())
        for x, y in zip((f.vertices, f.normals, f.colors), (m.vertices, m.normals, m.colors)):
            assert torch.equal(x, y[vi])
        g = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso, sparse=sparse,
                                min_component_faces=kw.get("min_faces", 0), largest_components=kw.get("largest"))
        if sparse:
            assert all(torch.equal(x, y) for x, y in zip(f, g))
        else:
            same_as_sets(f, g)


def test_defaults_change_nothing():
    h = hbr()
    enc, mlp, denc, mn, mx, _ = _field()
    iso = _iso(h, enc, mlp, mn, mx)
    a = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=192, iso=iso, sparse=True)
    b = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=192, iso=iso, sparse=True, min_component_faces=0,
                            largest_components=None)
    assert a.vertices.shape[0] > 0 and all(torch.equal(x, y) for x, y in zip(a, b))


def test_dense_and_sparse_agree_after_dropping_small_components():
    """Where every dense vertex the sparse route lost lies in a dense component with fewer than min_faces faces, the two
    filtered meshes are equal as sets.  That must hold on at least one case."""
    h = hbr()
    held = []
    for field, res in FIELD_CASES:
        enc, mlp, denc, mn, mx, _ = _field(coarse_only=field == "smooth")
        iso = _iso(h, enc, mlp, mn, mx)
        md = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso)
        ms = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso, sparse=True)
        nd = md.vertices.shape[0]
        label, fc, _ = cc.components(md.faces.cpu().numpy(), nd)
        both = torch.cat((md.vertices, ms.vertices)).contiguous().view(torch.int32)
        _, inv = torch.unique(both, dim=0, return_inverse=True)
        in_sparse = torch.zeros(int(inv.max()) + 1, device=DEV, dtype=torch.bool)
        in_sparse[inv[nd:]] = True
        lost = (~in_sparse[inv[:nd]]).cpu().numpy()
        lost_faces = int(fc[np.unique(label[lost])].max()) if lost.any() else 0
        for min_faces in (16, 256, 4096):
            if lost_faces >= min_faces:
                continue
            fd = h.mesh.filter_components(md, min_faces=min_faces)
            fs = h.mesh.filter_components(ms, min_faces=min_faces)
            assert fd.faces.shape[0] > 0
            same_as_sets(fd, fs)
            held.append((field, res, min_faces))
        print(f"{field} res={res}: {int(lost.sum())} dense vertices lost by the sparse route, in components of up to "
              f"{lost_faces} faces")
    print("dense == sparse after filtering:", held)
    assert held


def test_export_mesh_script_largest_component(tmp_path):
    h = hbr()
    from human_body_reconstruction_b200 import formats
    work = str(tmp_path)
    enc, mlp, _, mn, mx, _ = _field()
    iso = _iso(h, enc, mlp, mn, mx)
    formats.save_checkpoint(os.path.join(work, "s"), torch.nn.DataParallel(mlp.cpu()), enc.cpu())
    formats.save_bounds(os.path.join(work, "bounds_model.npy"), torch.tensor(mn), torch.tensor(mx))
    out = os.path.join(work, "mesh.ply")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "export_mesh.py"), "--ckpt_name", "s", "--bound_pth",
                        "bounds_model.npy", "--hash_size", "14", "--res", "160", "--iso", repr(iso), "--sparse",
                        "--largest-components", "1", "--out", out], cwd=work, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    rep = json.loads(r.stdout.strip().splitlines()[-1])
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import export_mesh
    e2, n2, d2, lo, hi = export_mesh.build_field(os.path.join(work, "s"), os.path.join(work, "bounds_model.npy"), 14, 2048.0)
    m = h.mesh.extract_mesh(e2, n2, d2, lo, hi, res=160, iso=iso, sparse=True)
    comp = h.mesh.mesh_components(m.faces, m.vertices.shape[0])
    f = h.mesh.filter_components(m, largest=1)
    back = h.mesh.read_ply(out)
    print(f"export: {rep['components']} components, {rep['components_kept']} kept, {rep['vertices']} of {m.vertices.shape[0]} "
          "vertices")
    assert rep["components"] == comp.roots.shape[0] > 1
    assert rep["components_kept"] == int(h.mesh.keep_components(comp, largest=1).sum()) >= 1
    assert back.vertices.shape[0] == f.vertices.shape[0] == rep["vertices"] < m.vertices.shape[0]
    assert back.faces.shape[0] == f.faces.shape[0] == rep["faces"]
    assert torch.equal(back.vertices, f.vertices.cpu()) and torch.equal(back.faces, f.faces.cpu())
    assert torch.equal(back.normals, f.normals.cpu())


def test_bounded_memory_at_2048_with_the_largest_component():
    """extract_mesh(sparse=True, largest_components=1) at 2048^3 stays within the sparse route's bound (the test in
    test_gpu_mesh_sparse.py) plus the labelling (3 x int32 per vertex) and the compaction (keep mask, prefix sum)."""
    h = hbr()
    from sparse_mc_oracle import brick_count
    enc, mlp, denc, mn, mx, _ = _field(coarse_only=True)
    iso = _iso(h, enc, mlp, mn, mx)
    res = 2048
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    m = h.mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso, sparse=True, largest_components=1)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    nv_kept = m.vertices.shape[0]
    del m
    surf = h.mesh.sparse_field_surface(enc, mlp, mn, mx, res, iso)
    n, nv, nf = surf.bricks.shape[0], surf.vertices.shape[0], surf.faces.shape[0]
    comp = h.mesh.mesh_components(surf.faces, nv)
    nb = brick_count(res)
    per_brick = max(2 * 729 * 4, 729 * 4 + 3 * 729 * 2) + 4 + 16
    bound = 4 * nb ** 3 + 4 * (nb + 1) ** 3 + n * per_brick + 12 * (nv + nf) + (1 << 19) * (6 + 128 + 4) + (64 << 20)
    bound += 12 * nv + 9 * nv
    print(f"2048^3 smooth field, largest component: {comp.roots.shape[0]} components, kept {nv_kept} of {nv} vertices "
          f"({nv_kept / nv:.4f}); peak {peak / 1e9:.2f} GB, bound {bound / 1e9:.2f} GB")
    assert 0 < nv_kept <= nv and peak <= bound
