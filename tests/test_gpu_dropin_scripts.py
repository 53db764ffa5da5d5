"""GPU tests (-m gpu): the reference's UNMODIFIED scripts run on the drop-in modules through launch.py.

train_hash2.py (the live trainer) and nerf2mesh.py are executed from oracle/_ref -- the verbatim copy of the reference
checkout that __graft_entry__.build() stages (or the checkout HBR_REFERENCE_DIR names); the scripts are not part of this
repository, so the tests skip where no copy was staged -- with launch.py building the import path (dropin/ in front of
the script directory).  Checked: the hot-path modules really came from dropin/, the sm_100a kernels
really ran (C-ABI call counters), and the files the scripts write (bounds_model.npy, *_Nerf_hash.pth, *_encoder_hash.pth,
density_grid_w_rgb.npy, the mesh) have the reference's names, keys and shapes.
"""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, load_golden, mlp_params
from oracle import port, ref_loader

pytestmark = pytest.mark.gpu
REF = ref_loader.REF_DIR
HAVE_REF = os.path.isfile(os.path.join(REF, "train_hash2.py"))
needs_ref = pytest.mark.skipif(not HAVE_REF, reason=f"runs the reference's own scripts: no reference copy at {REF} "
                               "(build() stages one where a reference checkout is present)")

RUNNER = r"""
import json, os, sys
sys.path.insert(0, {root!r})
import launch
try:
    launch.run({script!r}, {argv!r})
finally:
    from human_body_reconstruction_b200 import _lib
    mods = launch.served_by_dropin()
    with open({report!r}, "w") as f:
        json.dump({{"modules": mods, "calls": _lib.STATS.calls, "launches": _lib.STATS.launches}}, f)
"""


def run_script(script, argv, cwd, report, env=None, timeout=900):
    code = RUNNER.format(root=ROOT, script=os.path.join(REF, script), argv=list(argv), report=report)
    e = dict(os.environ)
    e.pop("PYTHONPATH", None)
    e.update(env or {})
    r = subprocess.run([sys.executable, "-c", code], cwd=cwd, env=e, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, f"{script} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    with open(report) as f:
        return json.load(f), r.stdout


@pytest.fixture(scope="module")
def trained(tmp_path_factory):
    """~20 steps of the unmodified train_hash2.py on the 2-view 5x6 scene (tests/golden/scene_new, the captured-humans
    json flavour), fp16 autocast + GradScaler as the script does, with --write so that it renders a test view and saves
    the checkpoints on its first iteration."""
    if not HAVE_REF:
        pytest.skip(f"no reference copy at {REF}")
    work = tmp_path_factory.mktemp("train")
    scene = os.path.join(work, "scene")
    shutil.copytree(os.path.join(GOLDEN, "scene_new"), scene)
    with open(os.path.join(scene, "transforms_train.json")) as f:
        meta = json.load(f)
    meta["frames"] = meta["frames"][:1]                  # train_hash2.py:55,279-293 renders ONE test view into an H*W buffer
    with open(os.path.join(scene, "transforms_tmp.json"), "w") as f:
        json.dump(meta, f)
    os.makedirs(os.path.join(work, "results"))
    rep, out = run_script("train_hash2.py", ["--data_path", scene + "/", "--num_epochs", "5", "--num_batch", "16", "--num_samples", "16",
                                             "--hash_size", "12", "--write", "--model_name", "m"], str(work),
                          os.path.join(work, "train_report.json"))
    return work, rep, out


@needs_ref
def test_train_hash2_runs_unmodified_on_the_dropins(trained):
    work, rep, out = trained
    # the hot-path modules came from dropin/, everything else (dataset_new.py, ...) from the reference
    for name in ("hash_encoding", "encoder", "test_hash", "helper", "vol_renderer", "tmp_encoder"):
        assert rep["modules"][name].startswith(os.path.join(ROOT, "dropin") + os.sep), name
    calls = rep["calls"]
    steps = 5 * 4                                        # 60 rays / 16 per batch = 4 batches per epoch, 5 epochs
    # train_hash2.py:218 runs torch.cuda.amp.autocast() = fp16: the tensor-core MLP kernels served every training step
    def n_calls(*names):                                 # the step's entry points changed names as kernels were fused
        return sum(calls.get(n, 0) for n in names)
    assert n_calls("hbr_mlp_fwd_tc") >= steps and n_calls("hbr_mlp_bwd_tc", "hbr_field_bwd_rays_tc") == steps
    assert n_calls("hbr_hash_encode_bwd", "hbr_hash_encode_bwd_rays", "hbr_field_bwd_rays_tc") == steps
    assert n_calls("hbr_hash_encode_fwd", "hbr_hash_encode_fwd_rays") >= steps
    assert n_calls("hbr_composite_bwd") == steps and n_calls("hbr_composite_fwd") >= steps
    assert "DATASET_LENGTH: 4" in out
    # files the script writes (train_hash2.py:115,299-300)
    b = np.load(os.path.join(work, "bounds_model.npy"))
    assert b.shape == (2, 3) and np.isfinite(b).all() and (b[0] < b[1]).all()
    nerf = torch.load(os.path.join(work, "m_Nerf_hash.pth"), map_location="cpu")
    encd = torch.load(os.path.join(work, "m_encoder_hash.pth"), map_location="cpu")
    want = [f"module.{n}.{i}.{w}" for n in ("sig_model", "col_model") for i in (0, 2, 4) for w in ("weight", "bias")]
    assert sorted(nerf.keys()) == sorted(want)
    # keys and shapes of the reference MLP_3D's own state_dict (tests/golden/mlp.npz, written by the unmodified reference)
    assert {k: tuple(v.shape) for k, v in nerf.items()} == {"module." + k: tuple(v.shape) for k, v in mlp_params(load_golden("mlp.npz")).items()}
    assert sorted(encd.keys()) == sorted(f"Embedding_list.{i}.weight" for i in range(16))
    assert all(tuple(v.shape) == (2 ** 12, 2) and v.dtype == torch.float32 for v in encd.values())
    assert all(torch.isfinite(v).all() for v in list(nerf.values()) + list(encd.values()))
    # the checkpoint loads into the REFERENCE's own classes (same keys / shapes), from the same staged copy as the script
    if ref_loader.available():
        ref = ref_loader.load()
        with ref_loader.quiet():
            e = ref.hash_encoding.HashEncoder(N_min=16, N_max=2048.0, L=16, F=2, T=2 ** 12, dim=3, mu=torch.zeros(3),
                                              sigma=torch.tensor(1.0), device="cpu")
            m = torch.nn.DataParallel(ref.test_hash.MLP_3D(num_sig=2, num_col=2, L=16, F=2, d_view=24,
                                                           max_bound=ref.Bound(torch.ones(3)), min_bound=ref.Bound(-torch.ones(3))))
        e.load_state_dict(encd)
        m.load_state_dict(nerf)


@needs_ref
def test_nerf2mesh_runs_unmodified_on_the_dropins(trained):
    """nerf2mesh.py on the checkpoint written above (density head shifted so that the iso level 30.0 is crossed): the
    256^3 density grid goes through the drop-in encoder / MLP per 400 000-point batch exactly as the script drives it, the
    mesh through dropin/torchmcubes.py (a CPU tensor in, as nerf2mesh.py:95-98 passes it)."""
    work, _, _ = trained
    mdir = os.path.join(work, "mesh")
    os.makedirs(mdir, exist_ok=True)
    nerf = torch.load(os.path.join(work, "m_Nerf_hash.pth"), map_location="cpu")
    encd = torch.load(os.path.join(work, "m_encoder_hash.pth"), map_location="cpu")
    # 20 steps from the U(-1e-4, 1e-4) table initialisation leave the density flat and near zero: give the field spatial
    # structure (trained-like table magnitudes, a steeper density head) centred on the script's iso level 30.0
    nerf["module.sig_model.4.weight"][0] *= 50.0
    nerf["module.sig_model.4.bias"][0] = nerf["module.sig_model.4.bias"][0] * 50.0 + 30.0
    torch.save(nerf, os.path.join(mdir, "s_Nerf_hash.pth"))
    torch.save({k: v * 1e4 for k, v in encd.items()}, os.path.join(mdir, "s_encoder_hash.pth"))
    shutil.copy(os.path.join(work, "bounds_model.npy"), os.path.join(mdir, "bounds_model.npy"))
    ply = os.path.join(mdir, "mesh.ply")
    rep, out = run_script("nerf2mesh.py", ["--ckpt_name", "s", "--bound_pth", "bounds_model.npy", "--hash_size", "12"], mdir,
                          os.path.join(mdir, "mesh_report.json"), env={"HBR_MESH_OUT": ply}, timeout=1500)
    for name in ("hash_encoding", "encoder", "helper", "torchmcubes"):
        assert rep["modules"][name].startswith(os.path.join(ROOT, "dropin") + os.sep), name
    calls = rep["calls"]
    n_batches = -(-256 ** 3 // 400000)
    assert calls.get("hbr_hash_encode_fwd", 0) == n_batches and calls.get("hbr_mlp_fwd_f32", 0) == n_batches
    assert calls.get("hbr_mc_count", 0) == 1 and calls.get("hbr_mc_emit", 0) == 1 and calls.get("hbr_grid_interp", 0) == 1
    grid = np.load(os.path.join(mdir, "density_grid_w_rgb.npy"))
    assert grid.shape == (256, 256, 256, 4) and np.isfinite(grid).all()
    # welded vertex count == iso-crossing grid edges of the saved density (the pinned marching-cubes invariant)
    head = []
    with open(ply) as f:
        for line in f:
            head.append(line)
            if line.startswith("end_header"):
                break
    nv = int([h for h in head if h.startswith("element vertex")][0].split()[-1])
    nf = int([h for h in head if h.startswith("element face")][0].split()[-1])
    assert nv == port.mc_crossing_edges(grid[..., 3], 30.0) and nv > 0 and nf > 0


@needs_ref
def test_train_hash2_use_sdf_runs_unmodified_on_the_sdf_kernels(tmp_path):
    """`train_hash2.py --use_sdf` (SURVEY 8f row 4), unmodified: VarModel + Volume_Renderer(use_sdf=True) as the script
    builds them (train_hash2.py:122-126; its MLP_3D keeps use_sdf=False, so the density column itself is composited as the
    SDF), the eikonal term in the loss (:223-224), three optimisers stepped through the GradScaler (:226-237).  Every step
    must go through the dedicated kernels of csrc/sdf.cu: one SDF compositing launch each way, one stencil, one eikonal
    launch each way -- and none through the NeRF-mode compositor."""
    work = str(tmp_path)
    scene = os.path.join(work, "scene")
    shutil.copytree(os.path.join(GOLDEN, "scene_new"), scene)
    shutil.copy(os.path.join(scene, "transforms_train.json"), os.path.join(scene, "transforms_tmp.json"))
    os.makedirs(os.path.join(work, "results"))
    rep, out = run_script("train_hash2.py", ["--data_path", scene + "/", "--num_epochs", "2", "--num_batch", "16", "--num_samples", "16",
                                             "--hash_size", "12", "--use_sdf", "--model_name", "s"], work,
                          os.path.join(work, "sdf_report.json"))
    assert rep["modules"]["helper"].startswith(os.path.join(ROOT, "dropin") + os.sep)
    calls, steps = rep["calls"], 2 * 4
    for name in ("hbr_composite_sdf_fwd", "hbr_composite_sdf_bwd", "hbr_sdf_stencil_points", "hbr_sdf_eikonal_fwd", "hbr_sdf_eikonal_bwd"):
        assert calls.get(name, 0) == steps, (name, calls)
    assert calls.get("hbr_composite_fwd", 0) == 0 and calls.get("hbr_mlp_fwd_tc", 0) == steps       # the field itself: fp16 autocast
    assert "DATASET_LENGTH: 4" in out


@needs_ref
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_train_hash2_unmodified_on_two_gpus(tmp_path):
    """torchrun + launch_rank.py: the unmodified trainer, one process per GPU; the drop-in renderer broadcasts rank 0's
    parameters and attaches the gradient all-reduce at its first call (HBR_AUTO_DP).  Both ranks must end with
    bit-identical checkpoints (same initial parameters, same averaged gradients every step)."""
    import socket
    work = str(tmp_path)
    scene = os.path.join(work, "scene")
    shutil.copytree(os.path.join(GOLDEN, "scene_new"), scene)
    with open(os.path.join(scene, "transforms_train.json")) as f:
        meta = json.load(f)
    meta["frames"] = meta["frames"][:1]
    with open(os.path.join(scene, "transforms_tmp.json"), "w") as f:
        json.dump(meta, f)
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port_no = sk.getsockname()[1]
    # every rank writes its own checkpoint: the model name carries the rank through a tiny wrapper around launch_rank
    wrapper = os.path.join(work, "rank_entry.py")
    with open(wrapper, "w") as f:
        f.write("import os, sys\n"
                f"sys.path.insert(0, {ROOT!r})\n"
                "rank = os.environ['RANK']\n"
                "os.makedirs(f'rank{rank}/results', exist_ok=True)\n"
                "os.chdir(f'rank{rank}')\n"
                "import launch_rank\n"
                "launch_rank.main()\n")
    e = dict(os.environ)
    e.pop("PYTHONPATH", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port_no), wrapper, os.path.join(REF, "train_hash2.py"), "--data_path", scene + "/",
           "--num_epochs", "3", "--num_batch", "16", "--num_samples", "16", "--hash_size", "12", "--write", "--model_name", "m"]
    r = subprocess.run(cmd, cwd=work, env=e, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    ck = [torch.load(os.path.join(work, f"rank{k}", "m_encoder_hash.pth"), map_location="cpu") for k in range(2)]
    nk = [torch.load(os.path.join(work, f"rank{k}", "m_Nerf_hash.pth"), map_location="cpu") for k in range(2)]
    # the checkpoint is written during the FIRST iteration (before its optimiser step): identical <=> the broadcast worked
    for key in ck[0]:
        assert torch.equal(ck[0][key], ck[1][key]), key
    for key in nk[0]:
        assert torch.equal(nk[0][key], nk[1][key]), key
