"""CPU: the connected-components oracle (tests/mesh_cc_oracle.py) against a plain union-find, the component selection rule
(mesh.keep_components), the stable compaction (mesh.filter_surface), and the input checks of ops.mesh_components, which
run before anything is launched."""
import numpy as np
import pytest
import torch

import mesh_cc_oracle as cc

from human_body_reconstruction_b200 import mesh, ops


def union_find(faces, nv):
    parent = list(range(nv))

    def find(x):
        while parent[x] != x:
            x = parent[x]
        return x

    for a, b, c in faces:
        for u, v in ((a, b), (a, c)):
            ru, rv = find(u), find(v)
            parent[max(ru, rv)] = min(ru, rv)
    label = np.array([find(v) for v in range(nv)], dtype=np.int64)
    fc = np.zeros(nv, dtype=np.int64)
    for a, _, _ in faces:
        fc[label[a]] += 1
    return label, fc, np.bincount(label, minlength=nv)


def random_mesh(nv, nf, seed, degenerate=True):
    rng = np.random.default_rng(seed)
    f = rng.integers(0, nv, (nf, 3))
    if degenerate and nf >= 4:
        f[0, 1] = f[0, 0]                                       # a == b
        f[1, 2] = f[1, 1]                                       # b == c
        f[2] = f[2, 0]                                          # a == b == c
    return f


@pytest.mark.parametrize("nv,nf,seed", [(1, 0, 0), (10, 0, 1), (50, 12, 2), (200, 60, 3), (300, 150, 4), (1000, 200, 5),
                                        (64, 400, 6)])
def test_oracle_matches_union_find(nv, nf, seed):
    f = random_mesh(nv, nf, seed)
    label, fc, vc = cc.components(f, nv)
    u_label, u_fc, u_vc = union_find(f.tolist(), nv)
    assert np.array_equal(label, u_label) and np.array_equal(fc, u_fc) and np.array_equal(vc, u_vc)
    assert (label <= np.arange(nv)).all() and np.array_equal(label[label], label)
    assert fc.sum() == nf and vc.sum() == nv
    roots, sf, sv = cc.sizes(label, fc, vc)
    used = np.zeros(nv, dtype=bool)
    used[f.reshape(-1)] = True
    assert np.array_equal(roots, np.unique(label)) and sf.sum() == nf and sv.sum() == nv
    assert (vc[~used] == (label[~used] == np.arange(nv)[~used])).all()          # an unused vertex is its own component


def test_oracle_empty():
    label, fc, vc = cc.components(np.zeros((0, 3), dtype=np.int64), 0)
    assert label.shape == fc.shape == vc.shape == (0,)


def comps(face_sizes):
    n = len(face_sizes)
    return mesh.MeshComponents(torch.zeros(0, dtype=torch.int32), torch.arange(n) * 10, torch.tensor(face_sizes, dtype=torch.int64),
                               torch.ones(n, dtype=torch.int64))


def test_keep_components_rule():
    c = comps([5, 40, 3, 40, 12, 0, 7])
    assert keep(c) == [True] * 7
    assert keep(c, min_faces=7) == [False, True, False, True, True, False, True]
    assert keep(c, largest=1) == [False, True, False, True, False, False, False]            # tied with the largest: both
    assert keep(c, largest=2) == [False, True, False, True, False, False, False]
    assert keep(c, largest=3) == [False, True, False, True, True, False, False]
    assert keep(c, largest=4) == [False, True, False, True, True, False, True]
    assert keep(c, largest=7) == keep(c, largest=100) == [True] * 7
    assert keep(c, min_faces=13, largest=3) == [False, True, False, True, False, False, False]
    assert keep(c, min_faces=1, largest=7) == [True, True, True, True, True, False, True]
    assert keep(comps([]), largest=1) == []
    c2 = comps([6, 6, 6, 2])
    assert keep(c2, largest=1) == [True, True, True, False]                                  # ties with the k-th all kept
    with pytest.raises(ValueError):
        mesh.keep_components(c2, largest=0)


def keep(c, **kw):
    return mesh.keep_components(c, **kw).tolist()


def test_keep_components_does_not_depend_on_order():
    rng = np.random.default_rng(0)
    sizes = rng.integers(0, 20, 200)
    for k in (1, 3, 17, 50):
        a = keep(comps(sizes.tolist()), largest=k, min_faces=4)
        p = rng.permutation(200)
        b = keep(comps(sizes[p].tolist()), largest=k, min_faces=4)
        assert np.array_equal(np.array(a)[p], np.array(b))


def test_filter_surface_is_a_stable_compaction():
    v = torch.arange(8 * 3, dtype=torch.float32).view(8, 3)
    f = torch.tensor([[0, 1, 2], [3, 4, 5], [2, 1, 6], [7, 6, 5], [6, 7, 2]], dtype=torch.int32)
    kv = torch.tensor([True, True, True, False, False, False, True, True])
    vi, f2 = mesh.filter_surface(v, f, kv)
    assert vi.dtype == torch.int64 and f2.dtype == torch.int32
    assert vi.tolist() == [0, 1, 2, 6, 7]
    assert f2.tolist() == [[0, 1, 2], [2, 1, 3], [3, 4, 2]]
    assert torch.equal(v[vi][f2.long()], v[f[[0, 2, 4]].long()])                 # the same triangles, in their order
    vi, f2 = mesh.filter_surface(v, f, torch.zeros(8, dtype=torch.bool))
    assert vi.shape == (0,) and f2.shape == (0, 3)
    with pytest.raises(ValueError):
        mesh.filter_surface(v, f, kv[:5])


def test_ops_need_cuda_without_a_device():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    f = torch.tensor([[0, 1, 2]], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mesh_components(f, 3)
    m = mesh.Mesh(torch.zeros(3, 3), f, torch.zeros(3, 3), torch.zeros(3, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        mesh.filter_components(m, largest=1)


@pytest.mark.parametrize("bad", [[[0, 1, 3]], [[0, -1, 2]], [[0, 1, 2], [5, 1, 2]], [[-7, 0, 0]]])
@pytest.mark.parametrize("dtype", [torch.int32, torch.int64])
def test_out_of_range_faces_raise_value_error(bad, dtype):
    with pytest.raises(ValueError, match="outside"):
        ops.mesh_components(torch.tensor(bad, dtype=dtype), 3)


def test_bad_shapes_and_sizes_raise_value_error():
    with pytest.raises(ValueError):
        ops.mesh_components(torch.zeros((4, 2), dtype=torch.int32), 3)
    with pytest.raises(ValueError):
        ops.mesh_components(torch.zeros((4, 3), dtype=torch.float32), 3)
    with pytest.raises(ValueError):
        ops.mesh_components(torch.zeros((0, 3), dtype=torch.int32), -1)
    with pytest.raises(ValueError):
        ops.mesh_components(torch.zeros((0, 3), dtype=torch.int32), 1 << 31)
    with pytest.raises(ValueError, match="outside"):
        ops.mesh_components(torch.tensor([[0, 0, 1 << 31]], dtype=torch.int64), 5)
