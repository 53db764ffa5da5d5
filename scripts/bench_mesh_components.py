"""Connected components of extracted meshes on one GPU (hbr_mesh_components) and floater removal in extract_mesh; prints ONE
JSON line (and writes it to --out).

Fields: bench_mesh_sparse.py's -- bench.py's grid leg ("busy") and the same with levels >= 4 zeroed ("smooth"), iso = the
median of the field's 64^3 grid.

1. Labelling: hbr_mesh_components (ops.mesh_components) on the 512^3 dense meshes, the 1024^3 sparse meshes and the 2048^3
   sparse mesh of the smooth field: CUDA-event time of each call after a warm-up, best and median of --reps (>= 5); the
   component count, the largest component's faces and vertices; an estimate of the bytes the four kernels move (faces
   read twice, labels and counts: 32 B per face + 24 B per vertex) and the rate it implies; the time of each of its four
   kernels in one profiled call (torch.profiler, outside the timed calls).  On the 512^3 meshes also
   scipy's connected_components host time over the same face edges (tests/mesh_cc_oracle.py), the CPU point of comparison.
2. extract_mesh(sparse=True) at 1024^3 and 2048^3 on the smooth field with and without largest_components=1: stage times
   (surface = sparse_field_surface, components = mesh.filter_by_components, attributes = index_surface_mesh), end to end
   (best of 3 after a warm-up), peak allocated memory above what was allocated before, vertices kept.

The device's name and power limit are read in the same run.

usage: python scripts/bench_mesh_components.py [--reps 7] [--out profiles/r06_bench_mesh_components.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_mesh import field  # noqa: E402
from bench_render import device_info  # noqa: E402
from human_body_reconstruction_b200 import mesh, ops  # noqa: E402

LABEL_RUNS = [(512, "busy", "dense"), (512, "smooth", "dense"), (1024, "busy", "sparse"), (1024, "smooth", "sparse"),
              (2048, "smooth", "sparse")]
EXTRACT_RUNS = [(1024, "smooth"), (2048, "smooth")]


def _ev():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def times_ms(fn, reps):
    fn()
    out = []
    for _ in range(reps):
        a = _ev()
        fn()
        b = _ev()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def surface(e, mlp, mn, mx, res, iso, route):
    if route == "sparse":
        s = mesh.sparse_field_surface(e, mlp, mn, mx, res, iso)
        return s.vertices, s.faces
    dens = mesh.density_grid(e, mlp, None, mn, mx, res)
    return mesh.marching_cubes(dens, iso)


def label_run(e, mlp, mn, mx, res, iso, route, reps):
    v, f = surface(e, mlp, mn, mx, res, iso, route)
    nv, nf = v.shape[0], f.shape[0]
    del v
    torch.cuda.empty_cache()
    t = times_ms(lambda: ops.mesh_components(f, nv), reps)
    comp = mesh.mesh_components(f, nv)
    big = int(torch.argmax(comp.faces))
    est = 32 * nf + 24 * nv
    r = {"vertices": nv, "faces": nf, "label_ms_best": min(t), "label_ms_median": statistics.median(t), "reps": reps,
         "components": int(comp.roots.shape[0]), "largest_faces": int(comp.faces[big]),
         "largest_vertices": int(comp.vertices[big]), "bytes_estimate": est, "estimate_GB_per_s_at_best": est / min(t) / 1e6}
    r["kernel_ms"] = kernel_split(lambda: ops.mesh_components(f, nv))
    if res <= 512:
        import mesh_cc_oracle
        fh = f.cpu().numpy()
        t0 = time.perf_counter()
        mesh_cc_oracle.components(fh, nv)
        r["scipy_host_s"] = time.perf_counter() - t0
    return r


def kernel_split(fn):
    """Device time of each of hbr_mesh_components' kernels in one call, from torch.profiler (a call of its own, not timed)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.key.split("(")[0].split("::")[-1]: getattr(e, "device_time_total", 0.0) / 1e3
            for e in prof.key_averages() if "cc_" in e.key}


def extract_stages(e, mlp, denc, mn, mx, res, iso, largest):
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    e0 = _ev()
    s = mesh.sparse_field_surface(e, mlp, mn, mx, res, iso)
    vidx, faces = s.vertices, s.faces
    del s
    e1 = _ev()
    comps = None
    if largest is not None:                    # extract_mesh's steps, one event between each
        vi, faces, comp, kept = mesh.filter_by_components(vidx, faces, 0, largest)
        nv_all = vidx.shape[0]
        vidx = vidx[vi]
        comps = (int(comp.roots.shape[0]), int(kept.sum()), nv_all)
        del comp, vi
    e2 = _ev()
    m = mesh.index_surface_mesh(e, mlp, denc, vidx, faces, mn, mx, res)
    e3 = _ev()
    torch.cuda.synchronize()
    r = {"largest_components": largest, "surface_ms": e0.elapsed_time(e1), "components_ms": e1.elapsed_time(e2),
         "attributes_ms": e2.elapsed_time(e3), "peak_GB": (torch.cuda.max_memory_allocated() - base) / 1e9,
         "vertices": int(m.vertices.shape[0]), "faces": int(m.faces.shape[0])}
    if comps:
        r.update(components=comps[0], components_kept=comps[1], kept_vertex_fraction=m.vertices.shape[0] / comps[2])
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be >= 5")
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh_components.py measures on a CUDA device")
    dev = torch.device("cuda", 0)
    line = {"bench": "mesh connected components and floater removal", **device_info(0)}
    enc, mlp, denc, mn, mx = field(dev)
    smooth = field(dev)[0]
    with torch.no_grad():
        for l, e in enumerate(smooth.Embedding_list):
            if l >= 4:
                e.weight.zero_()
    fields = {"busy": enc, "smooth": smooth}
    isos = {k: float(mesh.density_grid(e, mlp, None, mn, mx, 64).float().median()) for k, e in fields.items()}
    line.update(isos=isos, fields={"busy": "bench.py grid leg: T=2^19, N_max=2048, tables x2e5 (levels < 4) / x2e3",
                                   "smooth": "the same with levels >= 4 zeroed"})
    runs = []
    with torch.no_grad():
        for res, name, route in LABEL_RUNS:
            r = label_run(fields[name], mlp, mn, mx, res, isos[name], route, args.reps)
            r.update(res=res, field=name, route=route)
            runs.append(r)
            print(json.dumps(r), file=sys.stderr)
            torch.cuda.empty_cache()
        line["labelling"] = runs
        runs = []
        for res, name in EXTRACT_RUNS:
            e, iso = fields[name], isos[name]
            for largest in (None, 1):
                extract_stages(e, mlp, denc, mn, mx, res, iso, largest)                     # warm-up
                r = extract_stages(e, mlp, denc, mn, mx, res, iso, largest)
                torch.cuda.empty_cache()
                t = times_ms(lambda: mesh.extract_mesh(e, mlp, denc, mn, mx, res=res, iso=iso, sparse=True,
                                                       largest_components=largest), 3)
                r.update(res=res, field=name, extract_mesh_ms_best=min(t))
                runs.append(r)
                print(json.dumps(r), file=sys.stderr)
                torch.cuda.empty_cache()
        line["extract_mesh_sparse"] = runs
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
