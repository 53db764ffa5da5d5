"""Trained checkpoint -> oriented, coloured, world-space mesh as binary PLY.

Takes nerf2mesh.py's checkpoint flags and builds the modules as the trainer does (train_hash2.py:117-127,
nerf2mesh.py:56-65): HashEncoder(N_min=16, N_max=max_res, L=16, F=2, T=2**hash_size, dim=3, mu=min_bound,
sigma=|max_bound - min_bound|_2), PositionalEncoder(3, 4), MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24).  The
checkpoint loads through formats.load_checkpoint (with or without nn.DataParallel's `module.` prefix); the mesh comes
from mesh.extract_mesh and is written by mesh.write_ply (vertex x y z nx ny nz red green blue, faces counter-clockwise
seen from outside).  With --sparse the grid is evaluated and meshed only in the 8^3-cell bricks the surface passes through
(mesh.sparse_field_surface): memory and time follow the surface, so the field's finest resolution (--res 2048) fits; a
component that crosses no brick corner edge and never reaches a seeded brick is not meshed.  The JSON line then also
reports the active bricks and closure rounds.  --min-component-faces N / --largest-components K drop floaters (mesh
components with fewer than N faces / outside the K largest by face count, ties kept: mesh.keep_components) before the
normals and colours are computed; the JSON line then also reports the components before filtering and those kept.

usage: python scripts/export_mesh.py --ckpt_name NAME --bound_pth bounds_model.npy --hash_size 19
                                     [--max_res 2048] [--res 256] [--iso 30.0] [--sparse] [--min-component-faces N]
                                     [--largest-components K] [--out mesh.ply]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import human_body_reconstruction_b200 as hbr  # noqa: E402
from human_body_reconstruction_b200 import formats, mesh  # noqa: E402


def build_field(ckpt_name: str, bound_pth: str, hash_size: float, max_res: float, device="cuda"):
    """(encoder, nerf, dir_encoder, min_bound, max_bound) as the trainer builds them, weights from the checkpoint."""
    mn, mx = formats.load_bounds(bound_pth)
    min_bound, max_bound = torch.from_numpy(mn.copy()), torch.from_numpy(mx.copy())
    sigma = torch.linalg.vector_norm(max_bound - min_bound)
    enc = hbr.HashEncoder(N_min=16, N_max=max_res, L=16, F=2, T=int(2 ** hash_size), dim=3, mu=min_bound.to(device),
                          sigma=sigma.to(device), device=device)
    dir_enc = hbr.PositionalEncoder(3, 4)
    nerf = hbr.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=max_bound, min_bound=min_bound)
    formats.load_checkpoint(ckpt_name, nerf, enc, map_location="cpu")
    return enc.to(device), nerf.to(device), dir_enc, mn, mx


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--ckpt_name", required=True, help="checkpoint prefix: {name}_Nerf_hash.pth / {name}_encoder_hash.pth")
    ap.add_argument("--bound_pth", default="bounds_model.npy", help="the (2,3) [min_bound, max_bound] the trainer saved")
    ap.add_argument("--hash_size", type=float, default=19, help="log2 of the table size T the field was trained with")
    ap.add_argument("--max_res", type=float, default=2048.0, help="N_max of the hash encoder the field was trained with")
    ap.add_argument("--res", type=int, default=256, help="density-grid resolution per axis")
    ap.add_argument("--iso", type=float, default=30.0, help="density iso level of the surface")
    ap.add_argument("--sparse", action="store_true", help="mesh only the 8^3-cell bricks the surface passes through")
    ap.add_argument("--min-component-faces", type=int, default=0, help="drop mesh components with fewer faces")
    ap.add_argument("--largest-components", type=int, default=None,
                    help="keep only the K largest components by face count (ties with the K-th kept)")
    ap.add_argument("--out", default="mesh.ply", help="output PLY path")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("export_mesh.py needs a CUDA device")
    enc, nerf, dir_enc, mn, mx = build_field(args.ckpt_name, args.bound_pth, args.hash_size, args.max_res)
    t0 = time.perf_counter()
    extra = {}
    # extract_mesh's steps, spelled out for the counts the JSON line reports
    if args.sparse:
        surf = mesh.sparse_field_surface(enc, nerf, mn, mx, args.res, args.iso)
        extra = {"active_bricks": int(surf.bricks.shape[0]), "rounds": surf.rounds}
        vidx, faces = surf.vertices, surf.faces
        del surf
    else:
        dens = mesh.density_grid(enc, nerf, None, mn, mx, args.res)
        vidx, faces = mesh.marching_cubes(dens, args.iso)
        del dens
    if args.min_component_faces > 0 or args.largest_components is not None:
        vi, faces, comp, kept = mesh.filter_by_components(vidx, faces, args.min_component_faces, args.largest_components)
        vidx = vidx[vi]
        extra.update(components=int(comp.roots.shape[0]), components_kept=int(kept.sum()))
    m = mesh.index_surface_mesh(enc, nerf, dir_enc, vidx, faces, mn, mx, args.res)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    mesh.write_ply(args.out, m)
    t2 = time.perf_counter()
    print(json.dumps({"out": args.out, "vertices": int(m.vertices.shape[0]), "faces": int(m.faces.shape[0]),
                      "extract_s": t1 - t0, "write_s": t2 - t1, **extra}))


if __name__ == "__main__":
    main()
