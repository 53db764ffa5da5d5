#!/usr/bin/env python
"""bench.py -- headline measurement: train rays/s of one train_hash2.py-shaped step (hash encode -> field MLP ->
alpha compositing, forward + backward) on B200, through the reference-facing drop-in API.

    python bench.py --gpus 1 --steps 20 --warmup 5            # our arm (one JSON line)
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1   # the reference's algorithm on host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # weak scaling, rays sharded
    python bench.py --steps 20 --warmup 5 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy

A "step" = Volume_Renderer.vol_render(...) + MSE(Cr)+MSE(Cf) + loss.backward() on one batch of synthetic rays
(BASELINE.json configs[1]: 4096 rays x 128 samples, L=16 F=2 T=2^19, lego-shaped 800x800 scene).  The optimiser
step is not part of the metric (BASELINE.md section 3); gradient buffers are re-zeroed inside the step.

value   : rays/s with the ray batch already resident in HBM, timed with CUDA events per step, L2 flushed between
          steps (the 64 MiB table would otherwise sit in the 126 MB L2), max over ranks.
e2e     : same step driven from pinned HOST buffers: H2D of (rays_o, rays_d, dir_norm, gt) and a D2H read of the
          loss inside the timed region, wall clock.
roofline: the dominant kernel's algorithmic bytes / its mean CUDA-event duration inside the timed steps.
legs    : further sub-records of the same line, each skippable: c3 (configs[2]: 2^20 rays/step over the ranks, 2^17 at N=1;
          --no-c3), grid (configs[3]: 512^3 density grid + marching cubes, slabs over the ranks; --no-grid), c5 (configs[4]:
          T=2^22, 256 samples/ray hierarchical, N=1 only; --no-c5), occupancy_grid (--no-occupancy), device_sampler_e2e
          (--no-device-sampler), grad_check (N>1), cpu_baseline (N=1; --no-cpu-baseline).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic bytes per sample point (SURVEY.md section 8d), L=16 F=2 fp32
# (the _rays entry points are the same kernels fed from the rays; they are accounted with the survey's figures although
#  they move less: no 12-byte position read, 64-byte 16-bit feature rows instead of 128 -- the contract fixes the numerator)
BYTES_PER_POINT = {
    "hbr_hash_encode_fwd": 1164, "hbr_hash_encode_bwd": 1164, "hbr_hash_encode_fwd_rays": 1164, "hbr_hash_encode_bwd_rays": 1164,
    "hbr_hash_encode_fwd_pts": 1164, "hbr_hash_encode_bwd_pts": 1164, "hbr_mlp_fwd_f32": 144, "hbr_mlp_bwd_f32": 272,
    "hbr_mlp_fwd_tc": 144, "hbr_mlp_bwd_tc": 272, "hbr_composite_fwd": 16, "hbr_composite_bwd": 32,
    "hbr_field_fwd_tc": 1164 + 144, "hbr_field_fwd_rays_tc": 1164 + 144, "hbr_field_bwd_tc": 1164 + 272, "hbr_field_bwd_rays_tc": 1164 + 272,
}
# algorithmic FLOP per point of MLP_3D (SURVEY 8d): 27 904 forward, 2 x that for the backward GEMMs (dgrad + wgrad)
FLOPS_PER_POINT = {"hbr_mlp_fwd_tc": 27904, "hbr_mlp_bwd_tc": 55808, "hbr_mlp_fwd_f32": 27904, "hbr_mlp_bwd_f32": 55808}
STEP_BYTES_PER_POINT = 2792


def kernel_roofline(name, pts_per_launch, mean_ms, peaks):
    """Roofline entry of one C-ABI call: tensor-bound for the MLP GEMM chains, HBM-bound (effective bandwidth over the
    algorithmic bytes, gathers counted whether or not they hit L2) for everything else."""
    hbm, hbm_src, tf, tf_src = peaks
    if name in FLOPS_PER_POINT:
        ach = FLOPS_PER_POINT[name] * pts_per_launch / (mean_ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": name, "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf,
                "peak_source": tf_src, "algorithmic_flop_per_point": FLOPS_PER_POINT[name], "mean_launch_ms": mean_ms}
    ach = BYTES_PER_POINT.get(name, 0) * pts_per_launch / (mean_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
            "peak_source": hbm_src, "algorithmic_bytes_per_point": BYTES_PER_POINT.get(name), "mean_launch_ms": mean_ms}


# ---------------------------------------------------------------------------------------------------------------
# synthetic lego-shaped scene (SURVEY.md 8d): cameras on the upper hemisphere, radius 4.0311, looking at the origin
# ---------------------------------------------------------------------------------------------------------------
def make_cameras(n_views: int, seed: int = 0) -> torch.Tensor:
    rng = np.random.default_rng(seed)
    c2w = np.zeros((n_views, 4, 4), dtype=np.float32)
    for v in range(n_views):
        th = rng.uniform(0, 2 * np.pi)
        ph = rng.uniform(0.05, 0.5 * np.pi - 0.05)                      # elevation
        pos = 4.0311 * np.array([np.cos(ph) * np.cos(th), np.cos(ph) * np.sin(th), np.sin(ph)])
        z = pos / np.linalg.norm(pos)                                    # camera looks down -z (helper.py:201)
        x = np.cross([0, 0, 1.0], z)
        x /= np.linalg.norm(x)
        y = np.cross(z, x)
        c2w[v, :3, 0], c2w[v, :3, 1], c2w[v, :3, 2], c2w[v, :3, 3] = x, y, z, pos
        c2w[v, 3, 3] = 1
    return torch.from_numpy(c2w)


def intrinsics(H: int, W: int):
    focal = 0.5 * W / math.tan(0.5 * 0.6911112070083618)                # dataset.py:26
    K = torch.from_numpy(np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1]]))    # int64, train_hash2.py:67-72 (Q14)
    K[0, 0], K[1, 1], K[0, 2], K[1, 2] = focal, focal, W / 2, H / 2
    return K


def rays_for_pixels(c2w, K, view, px, py):
    """get_od (helper.py:176-208) evaluated for selected pixels only."""
    i = (px - K[0, 2]) / K[0, 0]
    j = (py - K[1, 2]) / K[1, 1]
    dirs = torch.stack((i, -j, -torch.ones_like(i)), dim=-1).float()
    R = c2w[view, :3, :3]
    d = torch.einsum("nij,nj->ni", R, dirs)
    n = torch.norm(d, dim=-1, keepdim=True)
    return c2w[view, :3, 3].clone(), d / n, n


def scene_bbox(c2w, K, H, W, near, far):
    """find_bounding_box (helper.py:109-141) over the image borders (the extremes of a pinhole frustum)."""
    xs = torch.arange(0, W, 8)
    ys = torch.arange(0, H, 8)
    px = torch.cat([xs, xs, torch.zeros_like(ys), torch.full_like(ys, W - 1)]).float()
    py = torch.cat([torch.zeros_like(xs), torch.full_like(xs, H - 1), ys, ys]).float()
    mn = torch.full((3,), 1e7)
    mx = torch.full((3,), -1e7)
    for v in range(c2w.shape[0]):
        o, d, _ = rays_for_pixels(c2w, K, torch.full((px.shape[0],), v, dtype=torch.long), px, py)
        for tt in (near, far + 1.5):
            p = o + d * tt
            mn, mx = torch.minimum(mn, p.min(0).values), torch.maximum(mx, p.max(0).values)
    return mx, mn


def make_batches(c2w, K, H, W, n_rays, n_batches, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_batches):
        view = torch.randint(0, c2w.shape[0], (n_rays,), generator=g)
        px = torch.randint(0, W, (n_rays,), generator=g).float()
        py = torch.randint(0, H, (n_rays,), generator=g).float()
        o, d, n = rays_for_pixels(c2w, K, view, px, py)
        gt = torch.stack([0.5 + 0.5 * torch.sin(px / 37.0), 0.5 + 0.5 * torch.cos(py / 23.0), (px + py) / (H + W)], dim=-1)
        out.append((o.contiguous(), d.contiguous(), n.contiguous(), gt.float().contiguous()))
    return out


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the measurement: an NVML polling thread (2 ms period -- the whole timed region
    of the default run lasts well under a second, so nvidia-smi's 100-200 ms loop alone yields a handful of samples),
    with the profiling recipe's `nvidia-smi --query-gpu=... -lms` loop as the fallback when NVML cannot be loaded."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    MASKS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.samples, self.stop_flag, self.thread = None, None, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        n, h = self.nvml, self.handle
        reasons_fn = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.samples.append((n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), int(reasons_fn(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            if not self.samples:
                return None
            sm = sorted(c for c, _ in self.samples)
            bits = 0
            for _, r in self.samples:
                bits |= r
            try:
                mx = self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)
            except Exception:
                mx = sm[-1]
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": [nm for nm, m in self.MASKS if bits & m],
                    "samples": len(sm), "source": "nvml, 2 ms period, median over the measurement"}
        if self.proc is None:
            return None
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        if not sm:
            return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k] == "Active" for r in self.rows)]
        mx = max(int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit())
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm), "source": "nvidia-smi -lms 100"}


def measured_peaks():
    """(HBM GB/s, source, bf16 TFLOP/s sustained -- the kernels are timed inside a long step --, source)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return (float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)",
                float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))), "measured sustained (MEASURED_PEAKS.json)")
    return 6650.0, "fallback (B200_PROFILING.md)", 1400.0, "fallback sustained (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference ITSELF (unmodified modules from the copy build() staged in oracle/_ref, loaded by
# oracle/ref_loader.py with environment shims only) on the box's host cores; oracle/port.py only when there is no copy.
# ---------------------------------------------------------------------------------------------------------------
def _reference_modules():
    from oracle import ref_loader
    return (ref_loader.load(), ref_loader) if ref_loader.available() else (None, ref_loader)


def reference_step(args, rays, device="cpu"):
    """Builds the reference's own objects the way train_hash2.py:117-127 does and returns (step_fn, kind, note):
    step_fn(k) runs vol_render + MSE(Cr)+MSE(Cf) + backward on batch k of the same synthetic scene as the B200 arm."""
    ref, ref_loader = _reference_modules()
    H = W = args.res
    c2w, K = make_cameras(args.views, 0), intrinsics(H, W)
    mx, mn = scene_bbox(c2w, K, H, W, args.near, args.far)
    sigma = ((mx - mn) ** 2).sum().sqrt()
    L, F, T = 16, 2, 2 ** args.hash_size
    batches = [tuple(t.to(device) for t in b) for b in make_batches(c2w, K, H, W, rays, 2, 100)]
    near, far = torch.tensor(args.near), torch.tensor(args.far)
    torch.manual_seed(0)
    if ref is None:
        from oracle import port
        g = torch.Generator().manual_seed(0)
        tables = ((torch.rand(L, T, F, generator=g) * 2 - 1)).requires_grad_()
        params = {k: v.requires_grad_() for k, v in port.mlp_init(seed=0).items()}
        scales = port.level_scales(16, float(args.max_res), L)

        def step(k):
            o, d, n, gt = batches[k % len(batches)]
            tt = port.strat_t(near, far, args.samples, torch.rand(args.samples))
            u_rs = torch.rand(rays, args.samples) if args.hierarchical else None
            u_s = torch.rand(args.samples) if args.hierarchical else None
            Cr, Cf, _ = port.vol_render(params, tables, mn, sigma, scales, d, o, tt, n, 4, args.hierarchical, near, far, u_rs, u_s)
            (torch.nn.functional.mse_loss(Cr, gt) + torch.nn.functional.mse_loss(Cf, gt)).backward()
            tables.grad = None
            for v in params.values():
                v.grad = None
        return step, "port", "oracle/port.py (torch-CPU restatement; no reference tree found on this box)"
    with ref_loader.quiet():
        enc = ref.hash_encoding.HashEncoder(N_min=16, N_max=float(args.max_res), L=L, F=F, T=T, dim=3, mu=mn.to(device),
                                            sigma=sigma.to(device), device=device)
        bound = (lambda t: t) if torch.cuda.is_available() else ref.Bound       # test_hash.py:25-26 calls .to('cuda')
        mlp = ref.test_hash.MLP_3D(num_sig=2, num_col=2, L=L, F=F, d_view=24, max_bound=bound(mx), min_bound=bound(mn))
        pe = ref.encoder.PositionalEncoder(3, 4)
    pe.sinus_in = pe.sinus_in.to(device)
    pe.device = device
    with torch.no_grad():
        for e in enc.Embedding_list:
            e.weight.mul_(1e4)                                            # trained-like magnitudes, as in the B200 arm
    enc, mlp = enc.to(device), mlp.to(device)
    vr = ref.vol_renderer.Volume_Renderer(H=H, W=W, K=K, near=near, far=far, device=device, Pos_encode=enc, Dir_encode=pe,
                                          max_dim=2 ** 10, sigma_val=sigma, mu=mn)
    params = list(enc.parameters()) + list(mlp.parameters())
    amp = device != "cpu"

    def step(k):
        o, d, n, gt = batches[k % len(batches)]
        for p in params:
            p.grad = None
        with ref_loader.quiet():
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):      # train_hash2.py:218 on the GPU; fp32 on the CPU
                Cr, Cf, _ = vr.vol_render(mlp, d, o, num_samples=args.samples, update_mask=False, dir_norm=n,
                                          hierarchical=args.hierarchical)
                loss = torch.nn.functional.mse_loss(Cr, gt) + torch.nn.functional.mse_loss(Cf, gt)
            (loss * (65536.0 if amp else 1.0)).backward()                       # GradScaler's initial scale (train_hash2.py:192,226)
    from oracle import ref_loader as rl
    return step, "reference", f"the unmodified reference modules from {rl.REF_DIR} (hash_encoding / encoder / test_hash / vol_renderer / helper)"


def cpu_reference_rays_per_s(args, steps, warmup, rays, budget_s=None):
    """Wall-clock rays/s of the reference's own CPU path, all host threads.  Returns (rays/s, s/step, kind, note, rays)."""
    torch.set_num_threads(os.cpu_count())
    if budget_s is not None:
        # keep the whole run inside the budget: time one small step first and shrink the per-step sample if 4096-ray steps
        # would not fit (the line then says so: cpu_baseline.sample / config.reference_rays_per_step)
        probe, _, _ = reference_step(args, 256)
        probe(0)
        t0 = time.perf_counter()
        probe(1)
        per_ray = (time.perf_counter() - t0) / 256
        while rays > 256 and per_ray * rays * (steps + warmup) > budget_s:
            rays //= 2
    step, kind, note = reference_step(args, rays)
    times = []
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        step(k)
        if k >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return rays / sec, sec, kind, note, rays


def workload_name(args, rays):
    return (f"train_hash2-shaped step: {rays} rays x {args.samples} samples/ray, L=16 F=2 T=2^{args.hash_size}, N_max={args.max_res}, "
            f"lego-shaped synthetic {args.res}x{args.res} x{args.views} views, hierarchical={args.hierarchical}, fwd+bwd "
            f"(encode+MLP+composite), no optimiser step")


def run_reference(args):
    """The reference arm: the reference's own implementation on the host cores, same scene / sizes / metric as the B200 arm.
    Each step is args.rays rays (the B200 arm's per-GPU batch) unless that cannot finish in a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm = max(args.warmup, 1)
    v, sec, kind, note, rays = cpu_reference_rays_per_s(args, args.steps, warm, args.rays, budget_s=args.reference_budget_s)
    line = {
        "impl": "reference", "metric": "train_rays_per_sec", "value": v, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, args.rays), "reference_rays_per_step": rays,
                   "same_rays_per_step_as_b200_arm": rays == args.rays},
        "cpu_baseline": {"value": v, "unit": "rays/s", "cores": os.cpu_count(), "kind": kind,
                         "sample": f"{rays} rays x {args.samples} samples per step of the same synthetic scene ({args.res}x{args.res} "
                                   f"views, T=2^{args.hash_size}), fwd+bwd, {note}, torch CPU fp32, {os.cpu_count()} threads"},
        "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


DUMP_ROWS = 1 << 17


def _dump_sample(x, dim):
    """x cut to a fixed seeded sample of DUMP_ROWS indices (ascending) along dim; whole when it has no more."""
    n = x.shape[dim]
    if n <= DUMP_ROWS:
        return x
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    return x.index_select(dim, idx.to(x.device))


def dump_outputs(path, outputs, enc, mlp):
    """--dump-outputs: what the last timed step hands its caller -- the loss, the colours of both passes and the parameter
    gradients -- as float32 DIR/<name>.npy.  Colours keep a fixed seeded sample of DUMP_ROWS rays and the table gradient
    (L, T, F) one of DUMP_ROWS table rows (the same rows on every level), so that the files stay far below 64 MB."""
    arrays = {"loss": outputs["loss"].reshape(1), "rgb_coarse": _dump_sample(outputs["rgb_coarse"], 0),
              "rgb_fine": _dump_sample(outputs["rgb_fine"], 0),
              "grad.hash_tables": _dump_sample(torch.stack([e.weight.grad for e in enc.Embedding_list]), 1)}
    arrays.update({f"grad.{n}": p.grad for n, p in mlp.named_parameters()})
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import human_body_reconstruction_b200 as hbr
    from human_body_reconstruction_b200 import _lib, dist as hdist
    from human_body_reconstruction_b200.graph import default_loss
    import torch.distributed as tdist

    rank, world = hdist.init_from_env("nccl")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    H = W = args.res
    c2w, K = make_cameras(args.views, 0), intrinsics(H, W)
    mx, mn = scene_bbox(c2w, K, H, W, args.near, args.far)
    sigma = ((mx - mn) ** 2).sum().sqrt()
    L, F, T = 16, 2, 2 ** args.hash_size
    torch.manual_seed(0)                                                  # identical parameters on every rank
    enc = hbr.HashEncoder(N_min=16, N_max=float(args.max_res), L=L, F=F, T=T, dim=3, mu=mn.to(dev), sigma=sigma.to(dev))
    with torch.no_grad():
        for e in enc.Embedding_list:
            e.weight.mul_(1e4)                                            # trained-like magnitudes U(-1,1) (SURVEY 8d)
    mlp = hbr.MLP_3D(num_sig=2, num_col=2, L=L, F=F, d_view=24, max_bound=mx, min_bound=mn)
    enc, mlp = enc.to(dev), mlp.to(dev)
    nerf = torch.nn.DataParallel(mlp, device_ids=[local])                 # as train_hash2.py:127 does
    pe = hbr.PositionalEncoder(3, 4)
    near, far = torch.tensor(args.near), torch.tensor(args.far)
    vr = hbr.Volume_Renderer(H=H, W=W, K=K, near=near, far=far, device=dev, Pos_encode=enc, Dir_encode=pe, max_dim=2 ** 10,
                             sigma_val=sigma, mu=mn)
    if args.fuse_field:
        vr.fuse_field = True                                              # encoder + MLP in one kernel per direction
    if args.fuse_gather:
        from human_body_reconstruction_b200 import vol_renderer as _vrm
        _vrm.FUSE_GATHER = True                                           # hash-grid gather + MLP forward in one kernel (A/B)
    if args.no_fuse_scatter:
        from human_body_reconstruction_b200 import vol_renderer as _vrm
        _vrm.FUSE_SCATTER = False                                         # MLP backward and hash-grid scatter-add as two kernels
    from human_body_reconstruction_b200 import vol_renderer as _vrm
    _vrm.STREAM_LEVEL_MAJOR = args.peer_scatter == "lm"
    reducer = None
    # "--peer-chunks 2" = two equal level ranges; "--peer-chunks 4,8,12,14" = inner level boundaries (cheap coarse levels first)
    # auto: streamed above 2 ranks (NVLS multicast); at 2 ranks (peer loads/stores) a launch pair per chunk measured faster
    streamed = args.peer_exchange == "stream" or (args.peer_exchange == "auto" and world > 2)
    pcs = str(args.peer_chunks) if args.peer_chunks != "auto" else ("4" if streamed else "2")
    pc = [int(v) for v in pcs.split(",") if v != ""]
    peer_chunks = pc if len(pc) > 1 else (pc[0] if pc else 0)
    if world > 1:
        # the gradient exchange: "peer" = this package's one-kernel all-reduce over NVLink peer memory (csrc/comm.cu),
        # "nccl" = torch.distributed all_reduce calls, "auto" = peer unless a rank cannot set it up
        reducer = hdist.attach_grad_allreduce(enc, mlp, kind=args.allreduce, transport=args.peer_transport, ctas=args.peer_ctas,
                                              overlap=peer_chunks != 0, chunks=peer_chunks if peer_chunks else 1,
                                              streamed=streamed)
    rays = args.rays                                                       # per GPU (weak scaling)
    host = [tuple(t.pin_memory() for t in b) for b in make_batches(c2w, K, H, W, rays, 4, 100 + rank)]
    resident = [tuple(t.to(dev) for t in b) for b in host]
    params = list(enc.parameters()) + list(mlp.parameters())
    flush = torch.empty(512 * 1024 * 1024 // 4, device=dev) if args.l2 == "flush" else None
    amp = args.precision in ("bf16", "f16")
    amp_dtype = torch.float16 if args.precision == "f16" else torch.bfloat16
    if args.precision == "f16":
        mlp.tc_grad_scale = 65536.0                # fp16 operands: what GradScaler's initial scale does in train_hash2.py:192,226

    outputs = {}                                   # --dump-outputs: colours and loss of the last step (detached)

    def keep(Cr, Cf, loss):
        outputs.update(rgb_coarse=Cr.detach(), rgb_fine=Cf.detach(), loss=loss.detach())

    def step(batch):
        o, d, n, gt = batch
        for p in params:
            p.grad = None
        with torch.autocast("cuda", dtype=amp_dtype, enabled=amp):
            Cr, Cf, _ = vr.vol_render(nerf, d, o, num_samples=args.samples, update_mask=False, dir_norm=n,
                                      hierarchical=args.hierarchical)
            loss = default_loss(Cr, Cf, gt)                       # MSE(Cr) + MSE(Cf), train_hash2.py:221 (one fused kernel)
        loss.backward()
        if args.dump_outputs:
            keep(Cr, Cf, loss)
        return loss

    def graph_loss(Cr, Cf, gt):
        """default_loss; during the capture it also keeps the tensors that every replay writes colours and loss into (the
        eager warm-up passes of GraphedStep.capture() keep nothing)."""
        loss = default_loss(Cr, Cf, gt)
        if args.dump_outputs and torch.cuda.is_current_stream_capturing():
            keep(Cr, Cf, loss)
        return loss

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    for k in range(args.warmup):
        step(resident[k % len(resident)])
    barrier()
    clocks = ClockSampler(local)
    clocks.start()

    def timed_region(run_step):
        """K steps, one CUDA-event pair per step on the launching stream, L2 flushed between steps."""
        ev = []
        for k in range(args.steps):
            if flush is not None:
                flush.zero_()                                              # evict L2 (outside the timed events)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_step(k)
            e1.record()
            ev.append((e0, e1))
        barrier()
        return sum(a.elapsed_time(b) for a, b in ev)

    # (1) eager region: every C-ABI call bracketed by its own CUDA events -> per-kernel durations for the roofline
    _lib.STATS.reset()
    _lib.STATS.timing = True
    t_wall0 = time.perf_counter()
    eager_ms = timed_region(lambda k: step(resident[k % len(resident)]))
    wall = time.perf_counter() - t_wall0
    _lib.STATS.timing = False
    launches = _lib.STATS.launches
    kern = _lib.STATS.summary()

    # (2) the same step captured once in a CUDA graph and replayed (one launch per step instead of ~35)
    gs, graph_note = None, "eager"
    if args.graph in ("on", "auto"):
        try:
            from human_body_reconstruction_b200.graph import GraphedStep
            outputs.clear()                                                # nothing of an eager step is released mid-capture
            gs = GraphedStep(vr, nerf, params, rays, args.samples, args.hierarchical, dev, loss_fn=graph_loss, autocast=amp,
                             autocast_dtype=amp_dtype).capture()
            host_packed = [GraphedStep.pack_batch(*b, pin=True) for b in host]       # one H2D copy per step
            resident_packed = [p.to(dev) for p in host_packed]
            for k in range(3):
                gs(resident_packed[k % len(resident_packed)])
            barrier()
            graph_note = "cuda graph replay (vol_render + loss + backward captured once)"
        except Exception as e:                                             # noqa: BLE001  (report, fall back to eager)
            gs, graph_note = None, f"eager (graph capture failed: {type(e).__name__}: {e})"
            for p in params:
                p.grad = None
    # the headline region is repeated: median of `--repeats` regions of K steps each (every region is K steps, barrier +
    # synchronize on both sides); the spread says how far one 10 ms region can be trusted
    run = (lambda k: gs(resident_packed[k % len(resident_packed)])) if gs is not None else (lambda k: step(resident[k % len(resident)]))
    region_ms = sorted(timed_region(run) for _ in range(max(1, args.repeats)))
    dev_ms = region_ms[len(region_ms) // 2]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs, enc, mlp)      # before the steps below overwrite the gradients

    # (3) end to end: pinned host batch -> H2D -> step -> loss.item()
    e2e_s = 0.0
    for k in range(args.steps):
        if flush is not None:
            flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if gs is not None:
            loss = gs(host_packed[k % len(host_packed)])                  # one non-blocking copy from pinned memory + replay
        else:
            batch = tuple(t.to(dev, non_blocking=True) for t in host[k % len(host)])
            loss = step(batch)
        loss_val = loss.item()
        e2e_s += time.perf_counter() - t0
    # (4) 8f row 2: the batch comes from the device-resident views (no host batch, no H2D): ray ids drawn on the device
    #     -> hbr_ray_gen -> static graph inputs -> replay -> loss.item()
    sampler = None
    if world == 1 and gs is not None and not args.no_device_sampler:
        try:
            yy, xx = torch.meshgrid(torch.arange(H, device=dev, dtype=torch.float32),
                                    torch.arange(W, device=dev, dtype=torch.float32), indexing="ij")
            img = torch.stack([0.5 + 0.5 * torch.sin(xx / 37.0), 0.5 + 0.5 * torch.cos(yy / 23.0), (xx + yy) / (H + W)], dim=-1)
            img = (img * 255).round().to(torch.uint8).expand(args.views, H, W, 3).contiguous()   # 192 MB at 100 x 800 x 800
            ds = hbr.DeviceRayDataset(img, c2w, K, device=dev, batch_size=rays)
            gs2 = GraphedStep(vr, nerf, params, rays, args.samples, args.hierarchical, dev, autocast=amp, autocast_dtype=amp_dtype,
                              source=ds).capture()
            for _ in range(3):
                gs2()
            torch.cuda.synchronize()
            s_s = 0.0
            for k in range(args.steps):
                if flush is not None:
                    flush.zero_()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                loss_s = gs2().item()
                s_s += time.perf_counter() - t0
            sampler = {"value": rays * args.steps / s_s, "unit": "rays/s", "ms_per_step": s_s * 1e3 / args.steps,
                       "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4, "resident_view_bytes": img.numel() + c2w.numel() * 4,
                       "note": "ray ids drawn on the device -> hbr_ray_gen from the resident views -> step, all captured in ONE "
                               "cuda graph; timed: replay + loss.item()", "last_loss": loss_s}
            del img, ds, gs2
        except Exception as e:                                             # noqa: BLE001
            sampler = {"error": f"{type(e).__name__}: {e}"}
    # (5) per-kernel durations INSIDE the replayed graph: a further capture of the same step with an external CUDA event
    #     (an event-record node of the graph) on either side of every C-ABI call.  The eager region (1) brackets the calls
    #     with events too, but there the host needs ~1.1 ms to enqueue what the GPU runs in ~0.47 ms, so an interval also
    #     holds the wait for the launch to arrive; inside the graph it is the kernel (plus a node boundary).
    kern_graph, kern_graph_note = None, None
    if gs is not None and args.graph_kernel_times and world == 1:     # N>1: the eager region's events (the exchange kernel's
                                                                       # cross-rank barriers stay out of a third capture)
        try:
            _lib.STATS.reset()
            _lib.STATS.timing = True
            gst = GraphedStep(vr, nerf, params, rays, args.samples, args.hierarchical, dev, autocast=amp, autocast_dtype=amp_dtype).capture()
            _lib.STATS.timing = False
            for k in range(3):
                gst(resident_packed[k % len(resident_packed)])
            torch.cuda.synchronize()
            acc = {}
            for k in range(args.steps):
                if flush is not None:
                    flush.zero_()
                gst(resident_packed[k % len(resident_packed)])
                torch.cuda.synchronize()
                for name, ts in _lib.STATS.graph_times().items():
                    c, tot = acc.get(name, (0, 0.0))
                    acc[name] = (c + len(ts), tot + sum(ts))
            kern_graph = {k: (c, tot / c) for k, (c, tot) in acc.items() if c}
            del gst
        except Exception as e:                                             # noqa: BLE001  (keep the eager figures)
            kern_graph, kern_graph_note = None, f"{type(e).__name__}: {e}"[:200]
        finally:
            _lib.STATS.timing = False
    barrier()
    clk = clocks.stop()

    tms = torch.tensor([dev_ms, e2e_s * 1e3, region_ms[0], region_ms[-1]], device=dev, dtype=torch.float64)
    if world > 1:
        tdist.all_reduce(tms, op=tdist.ReduceOp.MAX)
    dev_ms, e2e_ms, lo_ms, hi_ms = (float(v) for v in tms)
    occ = occupancy_leg(args, dev, vr, nerf, params, rays, resident_packed if gs is not None else None, flush, amp, amp_dtype,
                        mn, sigma) if (world == 1 and amp and gs is not None and not args.no_occupancy) else None
    c3 = c3_leg(args, world, rank, dev, vr, nerf, enc, mlp, params, c2w, K, H, W, amp, amp_dtype, barrier) if args.c3 else None
    grad_check = grad_check_leg(hdist, tdist, reducer, enc, mlp, params, step, resident, world, rank, args) if world > 1 else None
    grid = grid_leg(args, hbr, hdist, world, rank, dev, mx, mn, sigma, barrier) if args.grid else None
    c5 = c5_leg(args, hbr, dev, pe, mn, mx, sigma, near, far, flush, amp_dtype) if (world == 1 and amp and args.c5) else None
    if rank != 0:
        _finish(world)
        return
    pts_per_ray = args.samples * (3 if args.hierarchical else 1)
    n_pts = rays * pts_per_ray
    total_rays = rays * world * args.steps
    value = total_rays / (dev_ms / 1e3)
    peaks = measured_peaks()
    peak = peaks[0]
    # dominant kernel; durations from inside the replayed graph when that measurement succeeded, else from the eager region
    kern_eager = kern
    timing_src = "cuda events around every C-ABI call in the eager region (host-driven launches)"
    if kern_graph and all(k in kern_graph for k in kern if k in BYTES_PER_POINT or k in FLOPS_PER_POINT):
        kern = dict(kern_eager)
        kern.update(kern_graph)
        timing_src = "external cuda events recorded inside the replayed cuda graph, on either side of every C-ABI call"
    tot = {k: c * m for k, (c, m) in kern.items()}
    dom = max(tot, key=tot.get)
    traffic_tab = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic_tab = json.load(f)

    def roof(name):
        c, m = kern[name]
        r = kernel_roofline(name, n_pts / (c / args.steps), m, peaks)
        r["traffic"] = traffic_tab.get(name)       # dram bytes read+written per launch, one ncu --set full capture
        r["traffic_source"] = "imported from profiles/traffic.json (an earlier ncu --set full capture of this command), not measured in this run"
        r["timing"] = timing_src
        return r

    roofline = roof(dom)
    step_achieved = STEP_BYTES_PER_POINT * n_pts / (dev_ms / args.steps * 1e-3) / 1e9
    h2d = sum(t.numel() * t.element_size() for t in host[0])
    line = {
        "metric": "train_rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": f"{args.precision} MLP operands (f32 accumulate) / f32 encoder+compositor" if amp else "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args, rays), "rays_per_gpu": rays, "l2": "flushed between timed steps (512 MiB write)"
                   if flush is not None else "warm", "parallelism": f"dp{world} (rays sharded, table+MLP grads all-reduced)",
                   "launch": graph_note},
        "timed_regions": {"repeats": len(region_ms), "ms_per_step_median": dev_ms / args.steps, "ms_per_step_min": lo_ms / args.steps,
                          "ms_per_step_max": hi_ms / args.steps, "note": "each region = K steps between barrier+synchronize; value uses the median"},
        "eager_ms_per_step": eager_ms / args.steps,
        "e2e": {"value": total_rays / (e2e_ms / 1e3), "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches,
        "roofline": roofline,
        "kernel_rooflines": {k: {kk: vv for kk, vv in roof(k).items() if kk in ("bound", "achieved", "unit", "frac", "traffic")}
                             for k in sorted(kern) if k in BYTES_PER_POINT},
        "step_roofline": {"algorithmic_bytes_per_point": STEP_BYTES_PER_POINT, "achieved": step_achieved, "frac": step_achieved / peak,
                          "unit": "GB/s"},
        "kernels_ms": {k: {"launches_per_step": c / args.steps, "mean_ms": m} for k, (c, m) in sorted(kern_eager.items())},
        "kernels_ms_in_graph": ({k: {"launches_per_step": c / args.steps, "mean_ms": m} for k, (c, m) in sorted(kern_graph.items())}
                                if kern_graph else {"unavailable": kern_graph_note or "graph off"}),
        "eager_wall_ms_per_step_incl_flush": wall * 1e3 / args.steps,
        "clocks": clk, "last_loss": loss_val,
    }
    if "hbr_hash_encode_fwd" in kern:
        c, m = kern["hbr_hash_encode_fwd"]
        line["hash_encode_mpts_per_s"] = (n_pts / (c / args.steps)) / (m * 1e-3) / 1e6
    if sampler is not None:
        line["device_sampler_e2e"] = sampler
    if occ is not None:
        line["occupancy_grid"] = occ
    if c3 is not None:
        line["c3"] = c3
    if grad_check is not None:
        line["grad_check"] = grad_check
    if grid is not None:
        line["grid"] = grid
    if c5 is not None:
        line["c5"] = c5
    if reducer is not None:
        line["allreduce_bytes_per_step"] = 4 * sum(p.numel() for p in params)      # flat table + MLP gradients, fp32
        region = getattr(reducer, "region", None)
        line["config"]["allreduce"] = "nccl" if region is None else (
            f"one kernel over NVLink peer memory ({region.transport}{', NVLS multicast' if region.multicast_ptr else ''}"
            f"{f', overlapped level chunks {pcs}' if peer_chunks else ''}"
            f"{', streamed: one scatter-add launch + one exchange launch side by side' if getattr(reducer, 'streamed', False) else ''})")
        if region is not None and region.timed_out():
            line["error"] = "peer all-reduce barrier timed out"
    if world == 1 and not args.no_cpu_baseline:
        v, sec, kind, note, cr = cpu_reference_rays_per_s(args, 3, 1, args.cpu_rays)
        line["cpu_baseline"] = {"value": v, "unit": "rays/s", "cores": os.cpu_count(), "kind": kind,
                                "sample": f"{cr} rays x {args.samples} samples per step of the same synthetic scene, 1 warm-up + 3 timed "
                                          f"fwd+bwd steps of {note} (torch CPU fp32, {os.cpu_count()} threads)"}
        if args.reference_eager_b200:
            line["reference_eager_b200"] = reference_on_b200(args, rays)
    print(json.dumps(line), flush=True)
    _finish(world)


def occupancy_leg(args, dev, vr, nerf, params, rays, resident_packed, flush, amp, amp_dtype, mn, sigma):
    """SURVEY 8f row 3: the same step with the occupancy grid LIVE (Volume_Renderer.compact): a synthetic lego-sized
    object -- the cells whose centre lies in the cube |x|,|y|,|z| <= 1 around the origin the cameras look at -- is marked
    occupied, every sample outside it is skipped through encoder, MLP and compositor.  Graph replay, L2 flushed, CUDA events."""
    try:
        from human_body_reconstruction_b200.graph import GraphedStep
        G = vr.grid_size
        c = (torch.arange(G, device=dev, dtype=torch.float32) + 0.5) / G * float(sigma)
        ax = [c + float(mn[k]) for k in range(3)]
        inside = [(a.abs() <= 1.0) for a in ax]
        grid = inside[0][:, None, None] & inside[1][None, :, None] & inside[2][None, None, :]
        vr.bool_grid[...] = grid
        vr.compact = True
        from human_body_reconstruction_b200 import ops
        o, d = resident_packed[0][:3 * rays].view(rays, 3), resident_packed[0][3 * rays:6 * rays].view(rays, 3)
        t = torch.linspace(args.near, args.far, args.samples, device=dev)
        mu_h, sig_h = vr._norm_host()
        live = float(ops.compact_samples(o, d, t, vr.bool_grid, mu_h, sig_h)[3].item()) / (rays * args.samples)
        gs = GraphedStep(vr, nerf, params, rays, args.samples, False, dev, autocast=amp, autocast_dtype=amp_dtype)
        gs.load(resident_packed[0])
        gs.capture()
        for k in range(3):
            gs(resident_packed[k % len(resident_packed)])
        torch.cuda.synchronize()
        ev = []
        for k in range(args.steps):
            if flush is not None:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gs(resident_packed[k % len(resident_packed)])
            e1.record()
            ev.append((e0, e1))
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
        vr.bool_grid[...] = True
        vr.compact = False
        for p in params:
            p.grad = None
        return {"value": rays / (ms * 1e-3), "unit": "rays/s", "ms_per_step": ms, "occupied_cells_frac": float(grid.float().mean()),
                "live_samples_frac": live, "steps": args.steps,
                "note": "synthetic occupancy: cube |x|,|y|,|z| <= 1 around the scene centre marked occupied in the "
                        f"{G}^3 grid; samples outside are skipped (compacted lists); same rays, same step otherwise"}
    except Exception as e:                                                 # noqa: BLE001
        vr.bool_grid[...] = True
        vr.compact = False
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def c3_leg(args, world, rank, dev, vr, nerf, enc, mlp, params, c2w, K, H, W, amp, amp_dtype, barrier):
    """BASELINE configs[2]: 2^20 rays per step GLOBAL, sharded over the ranks (2^20 / N per GPU, table + MLP gradients
    all-reduced); at N = 1 the single-GPU rate is taken on 2^17 rays (what one of 8 GPUs processes).  Eager launches (the
    kernels run for milliseconds), 3 warm-up + 5 timed steps, CUDA events per step; reported: the median step, max over ranks."""
    import torch.distributed as tdist
    rays = (1 << 20) // world if world > 1 else 1 << 17
    try:
        b = make_batches(c2w, K, H, W, rays, 1, 7 + rank)[0]
        o, d, n, gt = (t.to(dev) for t in b)

        def step():
            for p in params:
                p.grad = None
            with torch.autocast("cuda", dtype=amp_dtype, enabled=amp):
                Cr, Cf, _ = vr.vol_render(nerf, d, o, num_samples=args.samples, update_mask=False, dir_norm=n, hierarchical=False)
                loss = 2.0 * torch.nn.functional.mse_loss(Cr, gt)
            loss.backward()
        for _ in range(3):
            step()
        barrier()
        nstep = 5
        evs = []
        for _ in range(nstep):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            evs.append((e0, e1))
        barrier()
        per_step = [a.elapsed_time(b) for a, b in evs]
        # median step of this rank, max over ranks: the eager step allocates ~10 GB of per-point temporaries and a single step
        # now and then pays a cudaMalloc of a fresh allocator segment (seen: one 76 ms step among four of 11.5 ms); the mean
        # and every step's time are reported beside it
        ms = torch.tensor([sorted(per_step)[nstep // 2], sum(per_step) / nstep], device=dev, dtype=torch.float64)
        if world > 1:
            tdist.all_reduce(ms, op=tdist.ReduceOp.MAX)
        ms, ms_mean = float(ms[0]), float(ms[1])
        del o, d, n, gt
        for p in params:
            p.grad = None
        torch.cuda.empty_cache()
        n_pts = rays * args.samples
        return {"workload": f"configs[2]: {rays * world} rays/step global = {rays} rays x {args.samples} samples per GPU on {world} GPU(s), "
                            f"T=2^{args.hash_size}, fwd+bwd" + (", gradients all-reduced" if world > 1 else " (single-GPU rate on 2^17 rays)"),
                "rays_global": rays * world, "rays_per_gpu": rays, "ms_per_step": ms, "value": rays * world / (ms * 1e-3), "unit": "rays/s",
                "steps": nstep, "warmup": 3, "launch": "eager", "ms_per_step_is": "median step, max over ranks", "ms_per_step_mean": ms_mean,
                "ms_each_step_this_rank": per_step,
                "step_roofline_frac_per_gpu": STEP_BYTES_PER_POINT * n_pts / (ms * 1e-3) / 1e9 / measured_peaks()[0]}
    except Exception as e:                                                 # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def c5_leg(args, hbr, dev, pe, mn, mx, sigma, near, far, flush, amp_dtype):
    """BASELINE configs[4], the human-reconstruction shape: T = 2^22 tables (512 MiB + 512 MiB of gradient), 256 samples per
    ray with hierarchical resampling (coarse 256 + fine 512 = 768 field evaluations per ray, both passes in the loss,
    train_hash2.py:221), 4096 rays of a 1080 x 1920 frame.  Graph replay, L2 flushed between steps, CUDA events; the step
    roofline is the same 2792 B per evaluated point."""
    try:
        from human_body_reconstruction_b200.graph import GraphedStep
        R, S, T = 4096, 256, 2 ** 22
        torch.manual_seed(5)
        enc = hbr.HashEncoder(N_min=16, N_max=args.max_res, L=16, F=2, T=T, dim=3, mu=mn.to(dev), sigma=sigma.to(dev))
        with torch.no_grad():
            for e in enc.Embedding_list:
                e.weight.mul_(1e4)
        mlp = hbr.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24, max_bound=mx, min_bound=mn)
        enc, mlp = enc.to(dev), mlp.to(dev)
        vr = hbr.Volume_Renderer(H=1080, W=1920, K=torch.eye(3), near=near, far=far, device=dev, Pos_encode=enc, Dir_encode=pe,
                                 max_dim=1024, sigma_val=sigma, mu=mn)
        g = torch.Generator().manual_seed(11)
        ro = (torch.tensor([[0.2, -0.1, 4.0]]).repeat(R, 1) + 0.05 * torch.randn(R, 3, generator=g)).to(dev)
        rd = torch.nn.functional.normalize(-ro.cpu() + 0.5 * torch.randn(R, 3, generator=g), dim=-1).to(dev)
        dn = (1 + 0.2 * torch.rand(R, 1, generator=g)).to(dev)
        gt = torch.rand(R, 3, generator=g).to(dev)
        params = list(enc.parameters()) + list(mlp.parameters())
        gs = GraphedStep(vr, mlp, params, R, S, True, dev, autocast=True, autocast_dtype=amp_dtype).capture()
        gs.load(ro, rd, dn, gt)
        for _ in range(3):
            gs()
        torch.cuda.synchronize()
        nstep, ev = 10, []
        for _ in range(nstep):
            if flush is not None:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gs()
            e1.record()
            ev.append((e0, e1))
        torch.cuda.synchronize()
        per = sorted(a.elapsed_time(b) for a, b in ev)
        ms = per[len(per) // 2]
        loss = float(gs.loss) if hasattr(gs, "loss") and torch.is_tensor(gs.loss) else None
        del gs, enc, mlp, vr, params
        torch.cuda.empty_cache()
        n_pts = R * 3 * S
        return {"workload": f"configs[4]: {R} rays x {S} samples/ray hierarchical (coarse {S} + fine {2 * S} evaluations per ray), "
                            f"L=16 F=2 T=2^22, fwd+bwd of both passes, synthetic 1080x1920 frame",
                "ms_per_step": ms, "ms_min": per[0], "ms_max": per[-1], "value": R / (ms * 1e-3), "unit": "rays/s", "steps": nstep,
                "warmup": 3, "launch": "cuda graph replay", "l2": "flushed between timed steps" if flush is not None else "warm",
                "points_per_step": n_pts, "last_loss": loss,
                "step_roofline_frac": STEP_BYTES_PER_POINT * n_pts / (ms * 1e-3) / 1e9 / measured_peaks()[0]}
    except Exception as e:                                                 # noqa: BLE001
        torch.cuda.empty_cache()
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def grid_leg(args, hbr, hdist, world, rank, dev, mx, mn, sigma, barrier):
    """BASELINE configs[3]: the nerf2mesh density-grid query (nerf2mesh.py:27-40,69-87) at 512^3 over the scene bounds plus
    marching cubes (:98), the grid sharded by slabs of its outermost axis over the ranks (each rank: its planes + one halo
    plane, vertices owned by the lower end point of each crossing edge, counts all-gathered).  Field: a smooth synthetic
    one (coarse hash levels only) so that the iso-surface looks like an object, not noise.  CUDA events, max over ranks."""
    import torch.distributed as tdist
    try:
        res, L, F, T = args.grid_res, 16, 2, 2 ** args.hash_size
        torch.manual_seed(1)
        enc = hbr.HashEncoder(N_min=16, N_max=float(args.max_res), L=L, F=F, T=T, dim=3, mu=mn.to(dev), sigma=sigma.to(dev))
        with torch.no_grad():
            for l, e in enumerate(enc.Embedding_list):
                e.weight.mul_(2e5 if l < 4 else 2e3)                     # smooth blobs: the coarse levels carry the shape
        mlp = hbr.MLP_3D(num_sig=2, num_col=2, L=L, F=F, d_view=24, max_bound=mx, min_bound=mn)
        enc, mlp = enc.to(dev), mlp.to(dev)
        lo, hi = mn.double().tolist(), mx.double().tolist()
        i0, i1 = hdist.slab_range(res, rank, world)
        halo = min(res, i1 + 1)

        def run():
            dens = hbr.mesh.density_grid(enc, mlp, None, lo, hi, res, i_begin=i0, i_end=halo)       # (planes + halo, res, res)
            return dens

        dens = run()
        # iso level: the median of the field on a coarse 64^3 grid over the same bounds -- every rank (and every N) computes
        # the same value, so the vertex / triangle totals are comparable across 1, 2, 4 and 8 GPUs
        iso = float(hbr.mesh.density_grid(enc, mlp, None, lo, hi, 64).float().median())
        barrier()
        ts, tc = [], []
        for _ in range(3):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            dens = run()
            e1.record()
            counts = hbr.ops.mc_count(dens, iso, 0, i1 - i0)               # vertices / triangles owned by this slab
            e2.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
            tc.append(e1.elapsed_time(e2))
        mine = [int(v) for v in counts.tolist()]
        allc = hdist.allgather_counts(mine)
        ms = torch.tensor([min(ts), min(tc)], device=dev, dtype=torch.float64)
        if world > 1:
            tdist.all_reduce(ms, op=tdist.ReduceOp.MAX)
        pts = res ** 3
        peak = measured_peaks()[0]
        roof_ms = 1034 * pts / world / (peak * 1e9) * 1e3
        out = {"workload": f"configs[3]: {res}^3 density grid over the scene bounds (fp16 positions, fp32 field: encoder + density head) "
                           f"+ marching-cubes count, {world} z-slab(s)", "density_ms": float(ms[0]), "mc_count_ms": float(ms[1]),
               "points": pts, "Mpts_per_s": pts / float(ms[0]) / 1e3, "roofline_ms_per_gpu": roof_ms, "frac": roof_ms / float(ms[0]),
               "algorithmic_bytes_per_point": 1034, "iso": iso, "vertices": sum(c[0] for c in allc), "triangles": sum(c[1] for c in allc),
               "per_rank_counts": allc}
        if world == 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            verts, faces = hbr.mesh.marching_cubes(dens, iso)
            e1.record()
            torch.cuda.synchronize()
            out["mc_emit_ms"] = e0.elapsed_time(e1)
            out["emitted"] = [int(verts.shape[0]), int(faces.shape[0])]
        del dens
        torch.cuda.empty_cache()
        return out
    except Exception as e:                                                 # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def grad_check_leg(hdist, tdist, reducer, enc, mlp, params, step, resident, world, rank, args):
    """N > 1: the reduced gradients are (a) bit-identical on every rank and (b) equal to the average of the ranks' LOCAL
    gradients, recomputed without the exchange on the same batches, on a sampled slice of every table level + the MLP."""
    try:
        L, T, F = enc.L, enc.T, enc.F
        idx = torch.randint(0, T, (256,), generator=torch.Generator().manual_seed(5)).to(enc._flat_table().device)

        def sample():
            tab = torch.stack([e.weight.grad for e in enc.Embedding_list])            # (L,T,F)
            return torch.cat([tab[:, idx, :].reshape(-1), torch.cat([p.grad.reshape(-1) for p in mlp.parameters()])]).clone()

        def checksum():
            tab = torch.stack([e.weight.grad for e in enc.Embedding_list])
            bits = torch.cat([tab.reshape(-1), torch.cat([p.grad.reshape(-1) for p in mlp.parameters()])]).view(torch.int32)
            return bits.to(torch.int64).sum().reshape(1)

        # the step draws its stratified depths from torch's generator (helper.strat_sampler): both passes start from the
        # same generator state so that they see the same samples
        torch.manual_seed(4242 + rank)
        step(resident[0])
        reduced, cs = sample(), checksum()
        all_cs = [torch.zeros_like(cs) for _ in range(world)]
        tdist.all_gather(all_cs, cs)
        identical = all(int(c) == int(all_cs[0]) for c in all_cs)
        if reducer is not None:
            reducer.remove()
        torch.manual_seed(4242 + rank)
        step(resident[0])                                                  # the same batch, gradients left local
        local = sample()
        gathered = [torch.zeros_like(local) for _ in range(world)]
        tdist.all_gather(gathered, local)
        want = torch.stack(gathered).double().mean(0)
        err = float((reduced.double() - want).norm() / (want.norm() + 1e-30))
        for p in params:
            p.grad = None
        return {"ranks_bit_identical": bool(identical), "rel_err_vs_recomputed_mean_of_local_grads": err, "ok": bool(identical and err < 1e-4),
                "sampled_entries": int(reduced.numel()), "note": "atomic accumulation order differs between the two backward passes: "
                "the comparison is norm-wise (1e-4), the rank-to-rank comparison is bit-exact"}
    except Exception as e:                                                 # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300], "ok": False}


def reference_on_b200(args, rays):
    """Second baseline (SURVEY 8c): the SAME unmodified reference modules run eagerly on this B200 (fp16 autocast as
    train_hash2.py:218), same scene and batch size.  Device-timed with CUDA events; a reported figure, not the target."""
    try:
        step, kind, note = reference_step(args, rays, device="cuda")
        if kind != "reference":
            return {"unavailable": "no reference tree on this box"}
        for k in range(2):
            step(k)
        torch.cuda.synchronize()
        n = 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(n):
            step(k)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        return {"value": rays / (ms * 1e-3), "unit": "rays/s", "ms_per_step": ms, "steps": n,
                "note": f"{note}, eager PyTorch on cuda:0, fp16 autocast, loss scaled by 65536, {rays} rays x {args.samples} samples"}
    except Exception as e:                                                 # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def _finish(world):
    """Multi-rank exit: everything is measured and printed; skip the process-group / CUDA-graph teardown (a graph that
    captured NCCL collectives keeps the communicator busy at destruction and can hang the interpreter exit)."""
    if world > 1:
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rays", type=int, default=4096, help="rays per GPU per step")
    ap.add_argument("--samples", type=int, default=128)
    ap.add_argument("--hash-size", type=int, default=19)
    ap.add_argument("--max-res", type=float, default=2048.0)
    ap.add_argument("--res", type=int, default=800)
    ap.add_argument("--views", type=int, default=100)
    ap.add_argument("--near", type=float, default=2.0)
    ap.add_argument("--far", type=float, default=6.0)
    ap.add_argument("--hierarchical", action="store_true")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "f16", "f32"],
                    help="MLP operand format: bf16 / f16 tensor-core kernels under autocast of that dtype, or the fp32 kernels")
    ap.add_argument("--l2", default="flush", choices=["flush", "warm"])
    ap.add_argument("--cpu-rays", type=int, default=1024, help="rays per step of the cpu_baseline leg of the B200 arm (bounded sample)")
    ap.add_argument("--reference-budget-s", type=float, default=300.0, help="--impl reference: shrink the per-step sample below "
                    "--rays only if (steps + warmup) full steps would not fit this many seconds")
    ap.add_argument("--reference-eager-b200", action="store_true", help="also time the unmodified reference modules eagerly on the GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-device-sampler", action="store_true", help="skip the device-resident ray sampler leg (8f row 2)")
    ap.add_argument("--allreduce", default="auto", choices=["auto", "peer", "nccl"], help="N>1 gradient exchange")
    ap.add_argument("--peer-transport", default="auto", choices=["auto", "ipc", "symm"])
    ap.add_argument("--peer-ctas", type=int, default=0)
    ap.add_argument("--peer-chunks", type=str, default="auto", help="> 0: all-reduce level chunks on a side stream while the "
                    "remaining chunks' scatter-add runs; 0: one all-reduce behind the backward pass; a list = inner level "
                    "boundaries; auto = 4 (streamed) / 2 (one launch per chunk)")
    ap.add_argument("--peer-scatter", default="tile", choices=["lm", "tile"], help="producer of the streamed exchange: the "
                    "level-major scatter-add (co-resident grid, levels in order) or the tile-major kernel launched chunk-major")
    ap.add_argument("--peer-exchange", default="auto", choices=["auto", "stream", "launch"], help="stream: ONE scatter-add launch "
                    "finishing the level chunks in order + ONE exchange launch beside it; launch: a launch pair per chunk")
    ap.add_argument("--fuse-field", action="store_true", help="use the fused encoder+MLP kernels (hbr_field_*_tc)")
    ap.add_argument("--fuse-gather", action="store_true", help="A/B: hbr_field_fwd_rays_tc, the hash-grid gather on dedicated "
                    "warps of the MLP forward kernel (measured slower than the two kernels: 152 vs 140 us)")
    ap.add_argument("--no-fuse-scatter", action="store_true", help="A/B: run the MLP backward and the hash-grid scatter-add as "
                    "two kernels (default on one GPU: hbr_field_bwd_rays_tc, the scatter-add on dedicated warps of the MLP kernel)")
    ap.add_argument("--no-grid", dest="grid", action="store_false", help="skip the configs[3] leg (512^3 density grid + marching cubes)")
    ap.add_argument("--grid-res", type=int, default=512)
    ap.add_argument("--no-occupancy", action="store_true", help="skip the live-occupancy-grid leg (8f row 3)")
    ap.add_argument("--repeats", type=int, default=5, help="timed regions of K steps each; value = their median")
    ap.add_argument("--no-graph-kernel-times", dest="graph_kernel_times", action="store_false",
                    help="skip the per-kernel timing inside the replayed graph (external event nodes); rooflines then use the eager region's events")
    ap.add_argument("--no-c5", dest="c5", action="store_false", help="skip the configs[4] leg (T=2^22, 256 samples/ray hierarchical; N=1 only)")
    ap.add_argument("--no-c3", dest="c3", action="store_false", help="skip the configs[2] leg (2^20 rays/step global; 2^17 at N=1)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step from a CUDA graph (auto = on; falls back to eager if capture fails)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (loss, "
                    "colours, parameter gradients; seeded samples of the large ones) as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device for the b200 arm (there is no CPU fallback)")
        run_b200(args)


if __name__ == "__main__":
    main()
