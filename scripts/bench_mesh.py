"""Mesh extraction on one GPU, stage by stage; prints ONE JSON line (and writes it to --out).

Field: bench.py's grid leg (the synthetic scene's bounds, T = 2^19, N_max = 2048, tables x 2e5 on levels < 4 and x 2e3
above), iso = the median of the 64^3 grid.  For each resolution (256 and 512): CUDA-event times of
  grid (density_grid, density only), mc (marching-cubes count + emit), world (index_to_world),
  normals = hash fwd + MLP fwd + bwd (density head, fp32) + dx kernel (hbr_hash_encode_dx), colours (dir_encode + full fp32 MLP),
  extract_mesh end to end,
then the host seconds of write_ply and the vertex / face counts.  Kernel timings of hbr_hash_encode_dx against
hash_fwd_kernel at 2^19 points and at the 512^3 vertex count, with effective GB/s by the algorithmic bytes (dx: 12 + 128 +
1 024 + 12 = 1 176 B/point; fwd: 1 164).  The device's name and power limit are read in the same run.

usage: python scripts/bench_mesh.py [--res 256 512] [--reps 5] [--out profiles/r04_bench_mesh.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402  (the synthetic scene of the benchmark)
import human_body_reconstruction_b200 as hbr  # noqa: E402
from bench_render import device_info  # noqa: E402
from human_body_reconstruction_b200 import mesh, ops  # noqa: E402

DX_BYTES, FWD_BYTES = 1176, 1164


def timed(fn, reps):
    """min over reps of CUDA-event ms around fn (one warm-up call first); returns (ms, last result)."""
    out = fn()
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best, out


def field(dev):
    c2w, K = bench.make_cameras(100, 0), bench.intrinsics(800, 800)
    mx, mn = bench.scene_bbox(c2w, K, 800, 800, 2.0, 6.0)
    sigma = ((mx - mn) ** 2).sum().sqrt()
    torch.manual_seed(1)
    enc = hbr.HashEncoder(N_min=16, N_max=2048.0, L=16, F=2, T=2 ** 19, dim=3, mu=mn.to(dev), sigma=sigma.to(dev))
    with torch.no_grad():
        for l, e in enumerate(enc.Embedding_list):
            e.weight.mul_(2e5 if l < 4 else 2e3)
    mlp = hbr.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=mx, min_bound=mn)
    return enc.to(dev), mlp.to(dev), hbr.PositionalEncoder(3, 4), mn.double().tolist(), mx.double().tolist()


def kernel_pair(x, enc, reps):
    """hbr_hash_encode_dx against the forward gather at the same N (fp32 positions); L2 is flushed between calls."""
    table, geom = enc._flat_table(), enc._geom()
    dy = torch.randn(x.shape[0], 32, device=x.device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=x.device)

    def run(fn):
        ts = []
        fn()
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    n = x.shape[0]
    t_dx = run(lambda: ops.hash_encode_dx(x, table, geom, dy))
    t_fw = run(lambda: ops.hash_encode_fwd(x, table, geom))
    return {"n": n, "dx_ms": t_dx, "fwd_ms": t_fw, "dx_effective_GBps": DX_BYTES * n / (t_dx * 1e-3) / 1e9,
            "fwd_effective_GBps": FWD_BYTES * n / (t_fw * 1e-3) / 1e9, "l2": "flushed (256 MB memset) before each call"}


def stages(enc, mlp, denc, mn, mx, res, iso, reps):
    table, geom = enc._flat_table(), enc._geom()
    params, dims = mlp._flat_params(), mlp._dims()
    out = {"res": res}
    out["grid_ms"], dens = timed(lambda: mesh.density_grid(enc, mlp, None, mn, mx, res), reps)
    out["mc_count_emit_ms"], (vidx, faces) = timed(lambda: mesh.marching_cubes(dens, iso), reps)
    del dens
    axes = mesh.world_axes(mn, mx, res, vidx.device)
    out["world_ms"], v = timed(lambda: mesh.index_to_world(vidx, axes), reps)
    n = v.shape[0]
    out["vertices"], out["faces"] = int(n), int(faces.shape[0])
    # normals and colours over all vertices in one pass each (extract_mesh's default chunk is 2^20: same kernels, more launches)
    out["normals_hash_fwd_ms"], feat = timed(lambda: ops.hash_encode_fwd(v, table, geom), reps)
    ones = torch.ones((n,), device=v.device)

    def mlp_fb():
        d, act = ops.mlp_fwd_f32(feat, None, 1, params, dims, keep_act=True)
        return ops.mlp_bwd_f32(feat, None, 1, params, dims, ones, act, True, False, None)[0]
    out["normals_mlp_fwd_bwd_ms"], dfeat = timed(mlp_fb, reps)
    out["normals_dx_ms"], g = timed(lambda: ops.hash_encode_dx(v, table, geom, dfeat), reps)
    out["normals_ms"] = out["normals_hash_fwd_ms"] + out["normals_mlp_fwd_bwd_ms"] + out["normals_dx_ms"]
    unit = g / g.norm(dim=1, keepdim=True).clamp_min(1e-30)

    def colours():
        return ops.mlp_fwd_f32(feat, ops.dir_encode(unit, denc.max_seq_len), 1, params, dims, keep_act=False)[0]
    out["colours_ms"], _ = timed(colours, reps)
    del feat, dfeat, g, unit, ones
    torch.cuda.empty_cache()
    out["extract_mesh_ms"], m = timed(lambda: mesh.extract_mesh(enc, mlp, denc, mn, mx, res=res, iso=iso), max(1, reps // 2))
    out["peak_GB"] = torch.cuda.max_memory_allocated() / 1e9
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        mesh.write_ply(os.path.join(d, "m.ply"), m)
        out["write_ply_s"] = time.perf_counter() - t0
        out["ply_MB"] = os.path.getsize(os.path.join(d, "m.ply")) / 1e6
    return out, v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh.py measures on a CUDA device")
    dev = torch.device("cuda", 0)
    line = {"bench": "mesh extraction", **device_info(0)}
    enc, mlp, denc, mn, mx = field(dev)
    iso = float(mesh.density_grid(enc, mlp, None, mn, mx, 64).float().median())
    line.update(iso=iso, field="bench.py grid leg: T=2^19, N_max=2048, tables x2e5 (levels < 4) / x2e3, fp32 field")
    runs, last_v = [], None
    for res in args.res:
        r, last_v = stages(enc, mlp, denc, mn, mx, res, iso, args.reps)
        runs.append(r)
        del r
        torch.cuda.empty_cache()
    line["stages"] = runs
    kp = [kernel_pair(torch.rand(1 << 19, 3, device=dev) * (torch.tensor(mx, device=dev) - torch.tensor(mn, device=dev)).float()
                      + torch.tensor(mn, device=dev).float(), enc, 2 * args.reps)]
    if last_v is not None:
        kp.append(kernel_pair(last_v, enc, 2 * args.reps))
    line["dx_kernel"] = kp
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
