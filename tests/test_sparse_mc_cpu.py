"""CPU: the numpy restatement of the sparse route's brick lattice (tests/sparse_mc_oracle.py) against a brick-by-brick
loop written from the definitions, and on hand-built volumes: a component inside one brick that no seed reaches is dropped,
closure travels along a tube for several rounds, res - 1 not a multiple of 8, and a single brick."""
import itertools

import numpy as np
import pytest

import sparse_mc_oracle as so
from oracle import port

B = so.B


def _grid(res):
    return np.meshgrid(*(np.arange(res, dtype=np.float64),) * 3, indexing="ij")


def _ball(res, c, r):
    """r - |p - c| (positive inside): float32."""
    i, j, k = _grid(res)
    return (r - np.sqrt((i - c[0]) ** 2 + (j - c[1]) ** 2 + (k - c[2]) ** 2)).astype(np.float32)


def two_components(res=64):
    """A ball around the coarse-lattice point (16,16,16) and a small ball inside brick (4,4,4), away from its planes."""
    return np.maximum(_ball(res, (16.0, 16.0, 16.0), 6.3), _ball(res, (36.2, 35.7, 36.4), 1.7))


def tube(res=65):
    """A tube along axis 0 at (j,k) = (5.3,5.6), radius 1.9, from i = 1 to i = 60, holding no coarse-lattice point, joined to
    a ball around (3,8,8) that holds the coarse point (0,8,8): only bricks at i < 8 are seeded, so closure must walk the tube
    brick by brick."""
    i, j, k = _grid(res)
    t = (1.9 - np.sqrt((j - 5.3) ** 2 + (k - 5.6) ** 2)) - np.maximum(0.0, i - 60.0) - np.maximum(0.0, 1.0 - i)
    return np.maximum(t.astype(np.float32), _ball(res, (3.0, 8.0, 8.0), 3.4))


def smooth(res, seed=0):
    """A sum of random Gaussian bumps (several components at iso 0.5)."""
    rng = np.random.default_rng(seed)
    i, j, k = _grid(res)
    v = np.zeros((res,) * 3)
    for _ in range(6):
        c = rng.uniform(0, res - 1, 3)
        s = rng.uniform(1.0, max(res / 5, 2.0))
        v += np.exp(-((i - c[0]) ** 2 + (j - c[1]) ** 2 + (k - c[2]) ** 2) / (2 * s * s))
    return v.astype(np.float32)


# ---- the definitions, brick by brick ------------------------------------------------------------------------------
def _brute(vol, iso):
    res = vol.shape[0]
    nb = so.brick_count(res)
    ins = vol < np.float32(iso)
    last = res - 1
    pts = {b: so.brick_points(res, b) for b in range(nb ** 3)}
    coords = {b: np.unravel_index(b, (nb, nb, nb)) for b in range(nb ** 3)}
    seeds = set()
    for b, Bc in coords.items():
        corner = [ins[min(B * (Bc[0] + d0), last), min(B * (Bc[1] + d1), last), min(B * (Bc[2] + d2), last)]
                  for d0, d1, d2 in itertools.product((0, 1), repeat=3)]
        if any(corner) and not all(corner):
            seeds.add(b)
    active, pending, rounds = set(), set(seeds), 0
    while pending:
        rounds += 1
        active |= pending
        new = set()
        for b in pending:
            i, j, k = pts[b]
            box = ins[np.ix_(i, j, k)]
            for a in range(3):
                for side in (0, 1):
                    nbc = list(coords[b])
                    nbc[a] += 1 if side else -1
                    if not 0 <= nbc[a] < nb:
                        continue
                    plane = np.take(box, 8 if side else 0, axis=a)
                    if plane.any() and not plane.all():
                        new.add(int(np.ravel_multi_index(nbc, (nb, nb, nb))))
        pending = new - active
    edges = set()
    for b in active:
        Bc = coords[b]
        for c in itertools.product(*[range(B * Bc[a], min(B * Bc[a] + B, last)) for a in range(3)]):
            for a in range(3):
                for o in itertools.product((0, 1), repeat=2):
                    p = list(c)
                    u, v = [x for x in range(3) if x != a]
                    p[u] += o[0]
                    p[v] += o[1]
                    q = list(p)
                    q[a] += 1
                    if ins[tuple(p)] != ins[tuple(q)]:
                        edges.add((tuple(p), a))
    iso32 = np.float32(iso)
    verts = []
    for p, a in edges:
        q = list(p)
        q[a] += 1
        d0, d1 = vol[p], vol[tuple(q)]
        x = np.array(p, dtype=np.float32)
        x[a] += (iso32 - d0) / (d1 - d0)
        verts.append(x)
    act = np.zeros(nb ** 3, dtype=bool)
    act[list(active)] = True
    return act.reshape((nb,) * 3), rounds, np.array(verts, dtype=np.float32).reshape(-1, 3)


@pytest.mark.parametrize("res,seed,iso", [(61, 0, 0.5), (25, 1, 0.4), (9, 2, 0.3), (5, 3, 0.5), (33, 4, 0.6)])
def test_oracle_matches_the_definitions_brick_by_brick(res, seed, iso):
    vol = smooth(res, seed)
    act, rounds = so.closure(vol, iso)
    b_act, b_rounds, b_verts = _brute(vol, iso)
    assert np.array_equal(act, b_act) and rounds == b_rounds
    assert np.array_equal(so.sorted_rows(so.crossing_vertices(vol, iso, act)), so.sorted_rows(b_verts))
    if res <= 9:
        assert act.shape == (1, 1, 1)


def test_component_inside_one_brick_is_dropped():
    vol = two_components()
    act, rounds = so.closure(vol, 0.0)
    dense = so.crossing_vertices(vol, 0.0)
    sparse = so.crossing_vertices(vol, 0.0, act)
    assert not act[4, 4, 4] and not so.covers_all_crossings(vol, 0.0, act)
    small = np.linalg.norm(dense - np.array([36.2, 35.7, 36.4]), axis=1) < 3
    assert small.sum() > 0
    assert len(sparse) == len(dense) - small.sum() == port.mc_crossing_edges(vol, 0.0) - small.sum()
    assert np.array_equal(so.sorted_rows(sparse), so.sorted_rows(dense[~small]))
    # the big ball is meshed whole: the triangles of the active cells are all the triangles outside brick (4,4,4)
    cells = np.zeros((63,) * 3, dtype=bool)
    cells[32:40, 32:40, 32:40] = True
    assert so.triangle_count(vol, 0.0, act) == so.triangle_count(vol, 0.0) - int(
        np.asarray(so.mc_tables.NUM_TRIS)[port.mc_case_index(vol, 0.0)][cells].sum())


def test_closure_walks_a_tube_for_several_rounds():
    vol = tube()
    seeds = so.seeds(vol, 0.0)
    act, rounds = so.closure(vol, 0.0)
    assert not seeds[2:, 0, 0].any()                        # the tube's far bricks are not seeded
    assert act[:8, 0, 0].all() and rounds >= 7
    assert so.covers_all_crossings(vol, 0.0, act)
    assert len(so.crossing_vertices(vol, 0.0, act)) == port.mc_crossing_edges(vol, 0.0)


def test_no_crossing_no_bricks():
    vol = smooth(61)
    act, rounds = so.closure(vol, 10.0)
    assert not act.any() and rounds == 0 and len(so.crossing_vertices(vol, 10.0, act)) == 0


def test_face_triples_compare_up_to_rotation_only():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    a = so.face_triples(v, np.array([[0, 1, 2]]))
    assert np.array_equal(a, so.face_triples(v, np.array([[1, 2, 0]])))
    assert not np.array_equal(a, so.face_triples(v, np.array([[0, 2, 1]])))            # the other winding
