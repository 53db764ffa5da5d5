"""Test support: the reference labelling of a triangle mesh's connected components (hbr.h, "connected components") --
scipy's connected_components over the face edges a-b, b-c, c-a, canonicalised to the smallest vertex index of each
component, with the sizes by the kernel's rules.  tests/test_mesh_components_cpu.py pins it against a plain union-find;
tests/test_gpu_mesh_components.py checks the kernel against it."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components


def components(faces, nv: int):
    """(label, face_count, vertex_count), int64 (nv,) each: label[v] = the smallest vertex index of v's component; the
    component's faces (a face counts for the component of its first vertex) and vertices at its root, 0 elsewhere."""
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    if nv == 0:
        return (np.zeros(0, dtype=np.int64),) * 3
    rows = np.concatenate((f[:, 0], f[:, 1], f[:, 2]))
    cols = np.concatenate((f[:, 1], f[:, 2], f[:, 0]))
    g = sp.coo_matrix((np.ones(len(rows), dtype=np.int8), (rows, cols)), shape=(nv, nv)).tocsr()
    _, comp = connected_components(g, directed=False)
    _, first = np.unique(comp, return_index=True)            # vertices ascend, so the first of each component is its minimum
    label = first[comp].astype(np.int64)
    return label, np.bincount(label[f[:, 0]], minlength=nv), np.bincount(label, minlength=nv)


def sizes(label, face_count, vertex_count):
    """(roots ascending, faces, vertices) of each component, int64 (C,)."""
    label = np.asarray(label)
    roots = np.nonzero(label == np.arange(len(label)))[0]
    return roots, np.asarray(face_count)[roots].astype(np.int64), np.asarray(vertex_count)[roots].astype(np.int64)
