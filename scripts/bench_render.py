"""Depth / opacity maps and whole-view rendering on one GPU; prints ONE JSON line.

  * render_view: rays/s for one 800 x 800 view of bench.py's synthetic scene (S = 128 coarse samples, hierarchical, T = 2^19,
    chunks of 2^16 rays), under fp16 autocast (the trainer's precision) and in fp32; median of --views-reps renders after
    one warm-up render, host clock around work that ends in a synchronize.
  * the C2 training step (bench.py's defaults: 4 096 rays x 128 samples, T = 2^19, bf16 tensor-core MLP), captured in a CUDA
    graph and replayed, L2 flushed between steps: vol_render + MSE (bench.py's step) against render + MSE + a depth term +
    binary cross-entropy of the opacity against a synthetic person mask, and render with the maps computed but the colour
    loss only (the compositor's own share).  The three are timed in alternating regions; the value is the median region.
  * the device's name and power limit, read in the same run.

usage: python scripts/bench_render.py [--steps 20] [--repeats 5] [--views-reps 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the synthetic scene and cameras of the benchmark)
import human_body_reconstruction_b200 as hbr  # noqa: E402
from human_body_reconstruction_b200.graph import GraphedStep, default_loss  # noqa: E402


def device_info(index: int) -> dict:
    info = {"device": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        pl, clk = [v.strip() for v in q.split(",")]
        info.update(power_limit=pl, max_sm_clock=clk)
    except Exception as e:                                                  # noqa: BLE001
        info.update(power_limit=f"not read ({type(e).__name__})")
    return info


def build_scene(res: int, hash_size: int, dev):
    H = W = res
    c2w, K = bench.make_cameras(100, 0), bench.intrinsics(H, W)
    mx, mn = bench.scene_bbox(c2w, K, H, W, 2.0, 6.0)
    sigma = ((mx - mn) ** 2).sum().sqrt()
    torch.manual_seed(0)
    enc = hbr.HashEncoder(N_min=16, N_max=2048.0, L=16, F=2, T=2 ** hash_size, dim=3, mu=mn.to(dev), sigma=sigma.to(dev))
    with torch.no_grad():
        for e in enc.Embedding_list:
            e.weight.mul_(1e4)                                              # trained-like magnitudes, as bench.py
    mlp = hbr.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=mx, min_bound=mn)
    enc, mlp = enc.to(dev), mlp.to(dev)
    nerf = torch.nn.DataParallel(mlp, device_ids=[dev.index])
    vr = hbr.Volume_Renderer(H=H, W=W, K=K, near=torch.tensor(2.0), far=torch.tensor(6.0), device=dev, Pos_encode=enc,
                             Dir_encode=hbr.PositionalEncoder(3, 4), max_dim=2 ** 10, sigma_val=sigma, mu=mn)
    return c2w, K, enc, mlp, nerf, vr


def map_loss(out, gt):
    """A depth term and a person-mask loss on the opacity: the mask is synthetic (blue channel of the target > 0.5)."""
    m = (gt[:, 2] > 0.5).float()
    a = out.opacity_fine.float().clamp(1e-4, 1 - 1e-4)
    bce = -(m * torch.log(a) + (1 - m) * torch.log(1 - a)).mean()
    return 1e-3 * out.depth_fine.float().mean() + bce


class MapsStep(GraphedStep):
    """GraphedStep with render() and the depth + mask terms in the loss."""
    with_map_loss = True

    def _step(self):
        with torch.autocast("cuda", dtype=self.autocast_dtype, enabled=self.autocast):
            out = self.renderer.render(self.model, self.rays_d, self.rays_o, num_samples=self.num_samples,
                                       dir_norm=self.dir_norm, hierarchical=self.hierarchical)
            loss = default_loss(out.rgb_coarse, out.rgb_fine, self.gt)
            if self.with_map_loss:
                loss = loss + map_loss(out, self.gt)
        loss.backward()
        return loss


class MapsUnused(MapsStep):
    """The maps kernels, but the colour loss only: what the compositor's maps cost by themselves."""
    with_map_loss = False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=800)
    ap.add_argument("--samples", type=int, default=128)
    ap.add_argument("--hash-size", type=int, default=19)
    ap.add_argument("--chunk", type=int, default=1 << 16)
    ap.add_argument("--views-reps", type=int, default=3)
    ap.add_argument("--rays", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_render.py needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    info = device_info(dev.index)
    c2w, K, enc, mlp, nerf, vr = build_scene(args.res, args.hash_size, dev)
    params = list(enc.parameters()) + list(mlp.parameters())

    # (1) render_view of one view
    n_px = args.res * args.res
    view = {}
    for name, amp in (("fp16_autocast", torch.float16), ("fp32", None)):
        times = []
        for k in range(args.views_reps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.autocast("cuda", dtype=amp or torch.float16, enabled=amp is not None):
                rgb, depth, opacity = vr.render_view(nerf, c2w[0], args.samples, hierarchical=True, chunk=args.chunk)
            torch.cuda.synchronize()
            if k:
                times.append(time.perf_counter() - t0)
        times.sort()
        s = times[len(times) // 2]
        view[name] = {"rays_per_s": n_px / s, "ms_per_view": s * 1e3, "ms_all": [round(v * 1e3, 2) for v in times],
                      "mean_opacity": float(opacity.mean()), "finite": bool(torch.isfinite(rgb).all() and torch.isfinite(depth).all())}
        del rgb, depth, opacity
    peak_mem = torch.cuda.max_memory_allocated(dev)

    # (2) the C2 step with and without the map terms, graph-replayed, alternating regions
    batches = bench.make_batches(c2w, K, args.res, args.res, args.rays, 4, 100)
    packed = [GraphedStep.pack_batch(*b).to(dev) for b in batches]
    flush = torch.empty(512 * 1024 * 1024 // 4, device=dev)
    steps = {}
    for name, cls in (("colour", GraphedStep), ("maps_colour_loss_only", MapsUnused), ("colour_depth_opacity", MapsStep)):
        gs = cls(vr, nerf, params, args.rays, args.samples, False, dev, autocast=True, autocast_dtype=torch.bfloat16)
        gs.load(packed[0])
        steps[name] = gs.capture()
    for gs in steps.values():
        for k in range(3):
            gs(packed[k % len(packed)])
    torch.cuda.synchronize()
    regions = {k: [] for k in steps}
    for _ in range(args.repeats):
        for name, gs in steps.items():
            ev = []
            for k in range(args.steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                gs(packed[k % len(packed)])
                e1.record()
                ev.append((e0, e1))
            torch.cuda.synchronize()
            regions[name].append(sum(a.elapsed_time(b) for a, b in ev) / args.steps)
    step = {}
    for name, r in regions.items():
        r = sorted(r)
        step[name] = {"ms_per_step": r[len(r) // 2], "min": r[0], "max": r[-1], "rays_per_s": args.rays / (r[len(r) // 2] * 1e-3),
                      "last_loss": float(steps[name].loss.detach())}
    step["delta_ms_maps_kernels"] = step["maps_colour_loss_only"]["ms_per_step"] - step["colour"]["ms_per_step"]
    step["delta_ms_map_loss"] = step["colour_depth_opacity"]["ms_per_step"] - step["colour"]["ms_per_step"]

    line = {"metric": "render_view_and_map_loss_step", **info,
            "render_view": {"res": [args.res, args.res], "samples": args.samples, "hierarchical": True, "T": 2 ** args.hash_size,
                            "chunk": args.chunk, "timing": "host clock around render_view, synchronized; median of "
                            f"{args.views_reps} after one warm-up", **view, "peak_memory_bytes": peak_mem},
            "c2_step": {"rays": args.rays, "samples": args.samples, "T": 2 ** args.hash_size, "precision": "bf16",
                        "timing": f"cuda graph replay, cuda events per step, L2 flushed; median of {args.repeats} alternating "
                                  f"regions of {args.steps} steps", **step}}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
