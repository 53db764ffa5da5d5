"""Sparse against dense mesh extraction on one GPU, stage by stage; prints ONE JSON line (and writes it to --out).

Fields: bench_mesh.py's (bench.py's grid leg: T = 2^19, N_max = 2048, tables x 2e5 on levels < 4 and x 2e3 above) --
"busy", detail everywhere -- and the same field with levels >= 4 zeroed -- "smooth" (as tests/test_gpu_mesh.py's
_field(coarse_only=True)).  iso = the median of the field's 64^3 grid.  Both routes at 512^3 and 1024^3 on both fields, the
sparse route alone at 2048^3 on the smooth field (the dense route would need 16 B x 2048^3 = 137 GB of grid and edge ids).

Per run, CUDA-event times of each stage -- dense: grid, mc, attributes (index_to_world + normals + colours); sparse: coarse
lattice, closure rounds (seed, compaction, brick field, closure steps), of which brick field, brick mc, attributes -- and
extract_mesh end to end (min over --reps after a warm-up); active bricks and their share of nb^3; field points evaluated
against res^3; peak allocated memory above what was allocated before the run; vertices and faces.  Where both routes ran: whether the meshes are identical (vertex
rows bitwise, faces as vertex triples up to rotation) and how many dense vertices the sparse route dropped.  The device's
name and power limit are read in the same run.

usage: python scripts/bench_mesh_sparse.py [--reps 3] [--out profiles/r05_bench_mesh_sparse.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_mesh import field  # noqa: E402
from bench_render import device_info  # noqa: E402
from human_body_reconstruction_b200 import mesh, ops  # noqa: E402

RUNS = [(512, "busy", ("dense", "sparse")), (512, "smooth", ("dense", "sparse")), (1024, "busy", ("dense", "sparse")),
        (1024, "smooth", ("dense", "sparse")), (2048, "smooth", ("sparse",))]


def _ev():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def best_ms(fn, reps):
    fn()
    best = float("inf")
    for _ in range(reps):
        a = _ev()
        fn()
        b = _ev()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def dense_stages(enc, mlp, denc, mn, mx, res, iso):
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    e0 = _ev()
    dens = mesh.density_grid(enc, mlp, None, mn, mx, res)
    e1 = _ev()
    vidx, faces = mesh.marching_cubes(dens, iso)
    e2 = _ev()
    del dens
    m = mesh.index_surface_mesh(enc, mlp, denc, vidx, faces, mn, mx, res)
    e3 = _ev()
    torch.cuda.synchronize()
    r = {"route": "dense", "grid_ms": e0.elapsed_time(e1), "mc_ms": e1.elapsed_time(e2), "attributes_ms": e2.elapsed_time(e3),
         "points": res ** 3, "peak_GB": (torch.cuda.max_memory_allocated() - base) / 1e9, "vertices": int(vidx.shape[0]),
         "faces": int(faces.shape[0])}
    return r, vidx, faces


def sparse_stages(enc, mlp, denc, mn, mx, res, iso):
    table, geom, params, dims = mesh._native_field(enc, mlp)
    field_ev = []

    def bricks(b):
        a = _ev()
        d = ops.brick_density(mn, mx, res, b, table, geom, params, dims)
        field_ev.append((a, _ev()))
        return d
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():                           # the stages of mesh.sparse_field_surface, one event between each
        e0 = _ev()
        coarse = ops.coarse_density(mn, mx, res, table, geom, params, dims)
        e1 = _ev()
        bmap, blist, dens, rounds = mesh.select_bricks(coarse, iso, bricks)
        e2 = _ev()
        vidx, faces = ops.brick_mc(dens, blist, bmap, res, iso)
        e3 = _ev()
        points = coarse.numel() + dens.numel()
        del dens, bmap, coarse
        m = mesh.index_surface_mesh(enc, mlp, denc, vidx, faces, mn, mx, res)
        e4 = _ev()
    torch.cuda.synchronize()
    nb = ops.brick_count(res)
    r = {"route": "sparse", "coarse_ms": e0.elapsed_time(e1), "closure_rounds_ms": e1.elapsed_time(e2),
         "brick_field_ms": sum(a.elapsed_time(b) for a, b in field_ev), "brick_mc_ms": e2.elapsed_time(e3),
         "attributes_ms": e3.elapsed_time(e4), "rounds": rounds, "active_bricks": int(blist.shape[0]), "bricks": nb ** 3,
         "active_fraction": blist.shape[0] / nb ** 3, "points": points, "points_fraction": points / res ** 3,
         "peak_GB": (torch.cuda.max_memory_allocated() - base) / 1e9, "vertices": int(vidx.shape[0]), "faces": int(faces.shape[0])}
    del m
    return r, vidx, faces


def _row_ranks(v):
    """rank of each vertex row in lexicographic order (stable sorts, last key first)."""
    order = torch.arange(v.shape[0], device=v.device)
    for c in (2, 1, 0):
        order = order[torch.sort(v[order, c], stable=True).indices]
    rank = torch.empty_like(order)
    rank[order] = torch.arange(v.shape[0], device=v.device)
    return order, rank


def _face_rows(f, rank):
    """faces as vertex ranks, rotated so the smallest rank leads (keeps the winding), rows sorted."""
    r = rank[f.long()]
    k = r.argmin(1, keepdim=True)
    r = torch.gather(r, 1, (k + torch.arange(3, device=r.device)) % 3)
    order = torch.arange(r.shape[0], device=r.device)
    for c in (2, 1, 0):
        order = order[torch.sort(r[order, c], stable=True).indices]
    return r[order]


def compare(dense, sparse):
    (vd, fd), (vs, fs) = dense, sparse
    od, rd = _row_ranks(vd)
    os_, rs = _row_ranks(vs)
    same_v = vd.shape == vs.shape and torch.equal(vd[od], vs[os_])
    same_f = same_v and fd.shape == fs.shape and torch.equal(_face_rows(fd, rd), _face_rows(fs, rs))
    return {"identical_mesh": bool(same_v and same_f), "dense_vertices_dropped": int(vd.shape[0] - vs.shape[0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh_sparse.py measures on a CUDA device")
    dev = torch.device("cuda", 0)
    line = {"bench": "sparse vs dense mesh extraction", **device_info(0)}
    enc, mlp, denc, mn, mx = field(dev)
    fields = {"busy": enc}
    smooth = field(dev)[0]
    with torch.no_grad():
        for l, e in enumerate(smooth.Embedding_list):
            if l >= 4:
                e.weight.zero_()
    fields["smooth"] = smooth
    isos = {k: float(mesh.density_grid(e, mlp, None, mn, mx, 64).float().median()) for k, e in fields.items()}
    line.update(isos=isos, fields={"busy": "bench.py grid leg: T=2^19, N_max=2048, tables x2e5 (levels < 4) / x2e3",
                                   "smooth": "the same with levels >= 4 zeroed"})
    runs = []
    for res, name, routes in RUNS:
        e, iso = fields[name], isos[name]
        meshes = {}
        for route in routes:
            stage = dense_stages if route == "dense" else sparse_stages
            stage(e, mlp, denc, mn, mx, res, iso)                                          # warm-up
            r, v, f = stage(e, mlp, denc, mn, mx, res, iso)
            torch.cuda.empty_cache()
            r["extract_mesh_ms"] = best_ms(lambda: mesh.extract_mesh(e, mlp, denc, mn, mx, res=res, iso=iso,
                                                                     sparse=route == "sparse"), args.reps)
            r.update(res=res, field=name)
            meshes[route] = (v, f)
            runs.append(r)
            print(json.dumps(r), file=sys.stderr)
            torch.cuda.empty_cache()
        if len(meshes) == 2:
            runs[-1].update(compare(meshes["dense"], meshes["sparse"]))
        del meshes
        torch.cuda.empty_cache()
    line["runs"] = runs
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
