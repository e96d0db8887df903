"""CPU-only: the parts of bench.py that run without a GPU keep their interface -- the reference arm prints one JSON
line with the agreed keys (rank 0 only), and the product arm refuses to run without a CUDA device (no CPU fallback).
GPU: --dump-outputs writes the maps the timed path computed."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH] + args, cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_the_contract_line():
    p = run(["--impl", "reference", "--workload", "C3", "--steps", "1", "--warmup", "0"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "disparity_volumes_per_s" and d["unit"] == "volumes/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["config"]["workload"].startswith("C3 synthetic 1280x720 D=64")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert "capped_8_threads" in cb and cb["capped_8_threads"]["cores"] <= 8     # MAX_CPU_THREADS, include/ComFunc.h:52
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    p = run(["--impl", "reference", "--workload", "C3", "--steps", "1", "--warmup", "0", "--gpus", "2"],
            env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_needs_the_product_path(tmp_path):
    for extra in (["--impl", "reference"], ["--emulate-shards", "2"]):
        p = run(["--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "out")] + extra)
        assert p.returncode != 0 and "--dump-outputs" in p.stderr
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_are_the_maps_of_the_timed_path(tmp_path):
    """--dump-outputs writes both disparity maps of the last timed step; they equal the maps the C-ABI gives
    for the same seeded frame."""
    import numpy as np
    from primestereomatch_b200 import DispEst, synth
    from bench import WORKLOADS
    p = run(["--workload", "C3", "--steps", "2", "--warmup", "0", "--no-cpu-baseline", "--no-parity",
             "--dump-outputs", str(tmp_path / "out")])
    assert p.returncode == 0, p.stderr[-2000:]
    W, H, D = WORKLOADS["C3"]
    l, r, _ = synth.stereo_pair_f32(W, H, D)
    with DispEst(l, r, D) as de:
        de.CostConst_GPU(); de.CostFilter_GPU(); de.DispSelect_GPU()
        want = {"lDisMap": de.lDisMap.copy(), "rDisMap": de.rDisMap.copy()}
    assert sorted(os.listdir(tmp_path / "out")) == ["lDisMap.npy", "rDisMap.npy"]
    for name, m in want.items():
        got = np.load(tmp_path / "out" / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == (H, W)
        assert np.array_equal(got, m.astype(np.float32)), name


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return  # on the GPU box the product arm is exercised by the driver itself
    p = run(["--steps", "1", "--warmup", "1", "--no-cpu-baseline"])
    assert p.returncode != 0
    assert "CUDA device" in (p.stderr + p.stdout)
