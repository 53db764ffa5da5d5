"""CPU: the reference arm of bench.py (`--impl reference`: the unmodified reference modules on host cores when
build() staged a copy of the reference in oracle/_ref, else the oracle port) prints ONE JSON line with the contract's keys,
labels the ray count it actually ran; under a multi-rank launch only rank 0 prints.
GPU: `--dump-outputs DIR` of the B200 arm writes what its last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


def _run(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--rays", "64", "--samples", "16", "--hash-size", "12", "--res", "64", "--views", "4",
                        "--gpus", env.get("WORLD_SIZE", "1")], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "train_rays_per_sec" and d["unit"] == "rays/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    from oracle import ref_loader
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_loader.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    # the label names what ran: 64 rays per step were asked for and fit the budget
    assert d["config"]["reference_rays_per_step"] == 64 and d["config"]["same_rays_per_step_as_b200_arm"] is True
    assert "64 rays x 16 samples" in d["config"]["workload"] and "64 rays x 16 samples" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    if isinstance(base.get("metric"), str):
        assert d["metric"] in base["metric"] or base["metric"] in d["metric"] or "rays" in base["metric"]


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


# T = 2^18 table rows: more than bench.DUMP_ROWS, so the table gradient is written as its seeded sample of rows
SMALL = ["--rays", "256", "--samples", "16", "--hash-size", "18", "--res", "64", "--views", "4", "--warmup", "1", "--repeats", "1",
         "--no-c3", "--no-grid", "--no-c5", "--no-occupancy", "--no-device-sampler", "--no-cpu-baseline", "--no-graph-kernel-times"]


def test_dump_sample_keeps_the_same_seeded_rows():
    """bench._dump_sample: an axis longer than DUMP_ROWS is cut to DUMP_ROWS distinct indices in ascending order, the same
    ones on every call and at every position of the other axes; a shorter one is kept whole."""
    import bench
    n = 2 * bench.DUMP_ROWS + 3
    rows = torch.arange(n, dtype=torch.float64)
    x = torch.stack([torch.stack([rows + 1e7 * l, rows + 1e7 * l + 0.5], dim=-1) for l in range(3)])     # (3, n, 2)
    s = bench._dump_sample(x, 1)
    assert s.shape == (3, bench.DUMP_ROWS, 2) and torch.equal(s, bench._dump_sample(x.clone(), 1))
    kept = s[0, :, 0]
    assert (kept[1:] > kept[:-1]).all() and 0 <= kept[0] and kept[-1] < n
    assert torch.equal(s, x[:, kept.long()])
    assert torch.equal(bench._dump_sample(x[:, :bench.DUMP_ROWS], 1), x[:, :bench.DUMP_ROWS])


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """float32 files within 64 MB; the same arguments give the same outputs (gradients up to the order of atomic
    additions; the sampled table gradient agrees only if both runs kept the same rows); --steps 2 and --steps 3 end on
    different ray batches, so their last steps differ."""
    import bench

    def dump(name, steps):
        d = str(tmp_path / name)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), *SMALL, "--dump-outputs", d],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64e6
        return {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}

    a, b, c = dump("a", 2), dump("b", 2), dump("c", 3)
    assert set(a) == set(b) == set(c)
    assert {"loss", "rgb_coarse", "rgb_fine", "grad.hash_tables", "grad.sig_model.0.weight", "grad.col_model.4.bias"} <= set(a)
    assert a["rgb_coarse"].shape == (256, 3) and a["grad.hash_tables"].shape == (16, bench.DUMP_ROWS, 2)
    assert np.linalg.norm(a["grad.hash_tables"]) > 0
    for k, v in a.items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        assert np.linalg.norm(v - b[k]) <= 1e-5 * np.linalg.norm(v) + 1e-12, k
    assert not np.allclose(a["rgb_coarse"], c["rgb_coarse"])
