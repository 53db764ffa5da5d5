"""Test support: numpy restatement of the sparse route's brick lattice (hbr.h, "sparse marching cubes") on a dense
(res, res, res) volume: the coarse lattice, seeds, face-plane closure to a fixpoint, and the vertex set marching cubes
gives over the active bricks' cells.  tests/test_sparse_mc_cpu.py checks it against a brick-by-brick loop and hand-built
volumes; tests/test_gpu_mesh_sparse.py checks the kernels against it."""
from __future__ import annotations

import numpy as np

from oracle import mc_tables, port

B = 8                                           # cells per brick and axis
P = B + 1


def brick_count(res: int) -> int:
    return -(-(res - 1) // B)


def lattice_index(res: int) -> np.ndarray:
    """Grid index of each coarse-lattice point along an axis: min(8c, res-1), c = 0..nb."""
    return np.minimum(B * np.arange(brick_count(res) + 1), res - 1)


def coarse(vol: np.ndarray) -> np.ndarray:
    ix = lattice_index(vol.shape[0])
    return vol[np.ix_(ix, ix, ix)]


def brick_points(res: int, b: int) -> np.ndarray:
    """(3, 9) grid indices of brick b's points along each axis, clamped to res-1."""
    nb = brick_count(res)
    Bc = np.array(np.unravel_index(b, (nb, nb, nb)))
    return np.minimum(B * Bc[:, None] + np.arange(P)[None], res - 1)


def brick_values(vol: np.ndarray, bricks) -> np.ndarray:
    """(n, 9, 9, 9) values of the listed bricks (brick-major, clamped indices)."""
    out = np.empty((len(bricks), P, P, P), dtype=vol.dtype)
    for s, b in enumerate(bricks):
        i, j, k = brick_points(vol.shape[0], int(b))
        out[s] = vol[np.ix_(i, j, k)]
    return out


def seeds(vol: np.ndarray, iso: float) -> np.ndarray:
    """(nb,nb,nb) bool: the 8 coarse values at a brick's corners straddle iso."""
    ins = coarse(vol) < np.float32(iso)
    n = sum(ins[dx:dx + ins.shape[0] - 1, dy:dy + ins.shape[1] - 1, dz:dz + ins.shape[2] - 1].astype(np.int32)
            for dx in (0, 1) for dy in (0, 1) for dz in (0, 1))
    return (n > 0) & (n < 8)


def _block_any(x: np.ndarray, axis: int, res: int) -> np.ndarray:
    """any over each brick's 9 points [8B, min(8B+8, res-1)] along `axis` of a boolean array."""
    starts = B * np.arange(brick_count(res))
    seg = np.logical_or.reduceat(x, starts, axis=axis)                 # [8B, 8B+8) (the last: [8B, res))
    nxt = np.take(x, np.minimum(starts + B, res - 1), axis=axis)
    return seg | nxt


def mixed_faces(vol: np.ndarray, iso: float):
    """For each axis a: (nb-1 along a, nb, nb) bool -- the 9x9 plane at grid index 8c (c = 1..nb-1) shared by bricks c-1
    and c holds values on both sides of iso."""
    res = vol.shape[0]
    nb = brick_count(res)
    ins = vol < np.float32(iso)
    out = []
    for a in range(3):
        planes = np.moveaxis(np.take(ins, B * np.arange(1, nb), axis=a), a, 0)       # (nb-1, res, res), other axes in order
        any_in = _block_any(_block_any(planes, 1, res), 2, res)
        any_out = _block_any(_block_any(~planes, 1, res), 2, res)
        out.append(np.moveaxis(any_in & any_out, 0, a))
    return out


def closure(vol: np.ndarray, iso: float):
    """(active (nb,nb,nb) bool, rounds): seeds, then round by round the face neighbours across mixed interior planes of the
    bricks evaluated last, until nothing is added.  rounds counts the evaluated batches (0 when there is no seed)."""
    faces = mixed_faces(vol, iso)
    pending = seeds(vol, iso)
    active = np.zeros_like(pending)
    rounds = 0
    while pending.any():
        rounds += 1
        active |= pending
        new = np.zeros_like(pending)
        for a in range(3):
            lo = [slice(None)] * 3
            hi = [slice(None)] * 3
            lo[a], hi[a] = slice(0, -1), slice(1, None)
            new[tuple(hi)] |= pending[tuple(lo)] & faces[a]                # brick c-1 -> c across plane 8c
            new[tuple(lo)] |= pending[tuple(hi)] & faces[a]                # brick c -> c-1
        pending = new & ~active
    return active, rounds


def _candidates(p: np.ndarray, a: int, nb: int):
    """The bricks (flat index) containing the edge from grid points p (N,3) along axis a, as up to 4 arrays in the owner
    order o, o-e_u, o-e_v, o-e_u-e_v, with a validity mask each."""
    u, v = [x for x in range(3) if x != a]
    o = np.minimum(p // B, nb - 1)
    su = (p[:, u] % B == 0) & (p[:, u] > 0) & (p[:, u] // B < nb)
    sv = (p[:, v] % B == 0) & (p[:, v] > 0) & (p[:, v] // B < nb)
    out = []
    for du, dv, ok in ((0, 0, np.ones_like(su)), (1, 0, su), (0, 1, sv), (1, 1, su & sv)):
        q = o.copy()
        q[:, u] -= du
        q[:, v] -= dv
        out.append((np.ravel_multi_index(tuple(np.clip(q, 0, nb - 1).T), (nb, nb, nb)), ok))
    return out


def crossing_vertices(vol: np.ndarray, iso: float, active=None) -> np.ndarray:
    """(V,3) float32 vertices of the crossing grid edges (all of them, or those in a cell of an active brick), in grid-index
    coordinates with hbr_mc_emit's float32 arithmetic: (float)i + (iso - d0) / (d1 - d0) along the edge axis."""
    res = vol.shape[0]
    nb = brick_count(res)
    iso32 = np.float32(iso)
    ins = vol < iso32
    rows = []
    for a in range(3):
        n_lo = [slice(None)] * 3
        n_hi = [slice(None)] * 3
        n_lo[a], n_hi[a] = slice(0, -1), slice(1, None)
        cross = ins[tuple(n_lo)] != ins[tuple(n_hi)]
        p = np.argwhere(cross)
        if active is not None and len(p):
            keep = np.zeros(len(p), dtype=bool)
            flat = active.reshape(-1)
            for b, ok in _candidates(p, a, nb):
                keep |= ok & flat[b]
            p = p[keep]
        d0 = vol[tuple(p.T)]
        q = p.copy()
        q[:, a] += 1
        d1 = vol[tuple(q.T)]
        t = (iso32 - d0) / (d1 - d0)
        xyz = p.astype(np.float32)
        xyz[:, a] += t
        rows.append(xyz)
    return np.concatenate(rows, 0).astype(np.float32)


def active_cells(res: int, active: np.ndarray) -> np.ndarray:
    """(res-1,)*3 bool: the cells of active bricks."""
    c = np.arange(res - 1) // B
    return active[np.ix_(c, c, c)]


def triangle_count(vol: np.ndarray, iso: float, active=None) -> int:
    """Triangles of the table over all cells (or the active bricks' cells)."""
    n = np.asarray(mc_tables.NUM_TRIS, dtype=np.int64)[port.mc_case_index(vol, float(np.float32(iso)))]
    if active is not None:
        n = n[active_cells(vol.shape[0], active)]
    return int(n.sum())


def covers_all_crossings(vol: np.ndarray, iso: float, active: np.ndarray) -> bool:
    """Every cell with a triangle lies in an active brick (then the sparse mesh is the dense mesh)."""
    n = np.asarray(mc_tables.NUM_TRIS)[port.mc_case_index(vol, float(np.float32(iso)))]
    return not (n[~active_cells(vol.shape[0], active)] > 0).any()


def sorted_rows(x: np.ndarray) -> np.ndarray:
    x = np.asarray(x)
    return x[np.lexsort(x.T[::-1])] if len(x) else x.reshape(0, x.shape[1] if x.ndim == 2 else 3)


def face_triples(verts: np.ndarray, faces: np.ndarray) -> np.ndarray:
    """(F, 9) sorted rows: each face as its three vertex coordinates in winding order, rotated to the lexicographically
    smallest of its three cyclic rotations (so faces compare up to rotation, keeping the winding)."""
    t = np.asarray(verts)[np.asarray(faces).astype(np.int64)]            # (F,3,3)
    F = len(t)
    if F == 0:
        return np.zeros((0, 9), dtype=np.float32)
    rot = np.stack([np.roll(t, -r, axis=1) for r in range(3)], 1).reshape(F * 3, 9)
    order = np.lexsort([rot[:, c] for c in range(8, -1, -1)] + [np.repeat(np.arange(F), 3)])
    return sorted_rows(rot[order[::3]])
