"""CPU: the parts of bench.py's contract that do not need a GPU - the reference arm (`--impl reference`, the CPU oracle
port) prints exactly ONE JSON line on stdout with the agreed keys, chatter goes to stderr, and under a multi-rank
launch only rank 0 prints."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CMD = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--lr", "32", "--batch", "2", "--steps", "1", "--warmup", "0"]


def run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run(CMD, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = run({"NCCL_DEBUG": "VERSION"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "oracle/femasr_oracle.py" in cb["sample"]
    assert d["config"]["workload"].startswith("config 2") and "model" not in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    r = run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_and_dump_outputs_arguments_are_checked():
    base = [sys.executable, os.path.join(ROOT, "bench.py")]
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run(base + extra, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 2 and r.stdout.strip() == "", (extra, r.stderr[-2000:])


def test_dump_samples_large_arrays_at_fixed_positions(tmp_path):
    import numpy as np
    import torch
    import bench
    n = bench.DUMP_MAX_VALUES + 8
    bench.dump_array(str(tmp_path / "a.npy"), torch.arange(n, dtype=torch.float64))
    bench.dump_array(str(tmp_path / "b.npy"), torch.arange(n, dtype=torch.int64).reshape(8, -1) * 2)
    pos, b = np.load(tmp_path / "a.npy"), np.load(tmp_path / "b.npy")
    assert pos.dtype == np.float64 and b.dtype == np.float32
    assert pos.ndim == 1 and 0 < pos.size <= bench.DUMP_MAX_VALUES and np.all(np.diff(pos) > 0)
    assert np.array_equal(b, 2 * pos)            # the same positions for every array of that size


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path, cuda):
    """--dump-outputs writes the forward's outputs for bench.py's seeded inputs, exactly as FeMaSRNet computes them."""
    import numpy as np
    import torch
    from basicsr.archs.femasr_arch import FeMaSRNet
    from femasr_b200.spec import random_state_dict
    B, S = 2, 64
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--lr", str(S), "--batch", str(B), "--steps", "2",
           "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert sorted(got) == ["codebook_loss", "indices", "sr"] and all(a.dtype == np.float32 for a in got.values())
    net = FeMaSRNet(codebook_params=[[32, 1024, 256]], LQ_stage=True, scale_factor=4)
    net.load_state_dict(random_state_dict(4, 256, seed=0, init="default"), strict=True)
    net = net.to(cuda).eval()
    x = torch.rand(B, 3, S, S, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        out, loss, _sem, idx = net(x.to(cuda))
    assert np.array_equal(got["sr"], out.cpu().numpy())
    assert np.array_equal(got["codebook_loss"], loss.cpu().numpy())
    assert np.array_equal(got["indices"], idx[0].cpu().numpy().astype(np.float32))
