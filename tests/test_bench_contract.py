"""bench.py contract checks that need no GPU: the reference arm (the unmodified reference from oracle/_ref, or the oracle port, timed on host cores) prints one JSON
line with the keys the driver reads, non-zero ranks of a multi-process launch stay silent, and the product arm refuses
to run without a CUDA device instead of falling back to anything on the CPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env_extra=None, timeout=600):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=env, timeout=timeout,
                          capture_output=True, text=True)


def test_reference_arm_prints_the_contract_line():
    res = _run(["--impl", "reference", "--workload", "cfg1", "--steps", "2", "--warmup", "1"])
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "region-timesteps/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    staged = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "STMGCN.py"))
    assert d["value"] > 0 and d["cpu_baseline"]["cores"] >= 1
    # the unmodified reference (staged by oracle/stage_reference.py) when present, else the oracle port
    assert d["cpu_baseline"]["kind"] == ("reference" if staged else "port")
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
    assert "workload" in d["config"]


def test_reference_arm_non_zero_rank_is_silent():
    res = _run(["--impl", "reference", "--workload", "cfg1", "--gpus", "2", "--steps", "1", "--warmup", "0"],
               {"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29577"})
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on a machine without a GPU")
def test_product_arm_refuses_to_run_without_cuda():
    res = _run(["--workload", "cfg1", "--steps", "1", "--warmup", "0", "--no-cpu-baseline"])
    assert res.returncode != 0
    assert "CUDA" in (res.stderr + res.stdout)


def test_steps_must_be_at_least_one():
    res = _run(["--impl", "reference", "--workload", "cfg1", "--steps", "0"])
    assert res.returncode != 0 and "--steps" in res.stderr


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: the output, loss and every parameter gradient of the last timed step, float32, inside 64 MB."""
    from stmgcn_b200 import synth
    res = _run(["--workload", "cfg1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
                "--dump-outputs", str(tmp_path)])
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2
    got = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype == np.float32 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    w = synth.WORKLOADS["cfg1"]
    _, y = synth.make_inputs(w, seed=100, batch=w.batch)
    assert got["out"].shape == tuple(y.shape)
    loss = float(got["loss"])
    assert abs(float(np.mean((got["out"].astype(np.float64) - y.numpy()) ** 2)) - loss) <= 1e-5 * loss
    # the loss check after the timing re-runs the same step on the same inputs
    assert abs(d["loss_check"]["loss"] - loss) <= 1e-5 * loss
    import STMGCN
    names = {"grad." + k for k, _ in STMGCN.ST_MGCN(**synth.model_kwargs(w)).named_parameters()}
    assert names == {k for k in got if k.startswith("grad.")}
    assert all(np.isfinite(got[k]).all() and np.abs(got[k]).max() > 0 for k in names)
    # --steps sets how many steps run in the timed region: the library launches counted over it, divided by --steps,
    # give the same launches per step for another --steps
    res5 = _run(["--workload", "cfg1", "--steps", "5", "--warmup", "1", "--no-cpu-baseline", "--no-e2e"])
    assert res5.returncode == 0, res5.stderr[-2000:]
    d5 = json.loads([l for l in res5.stdout.splitlines() if l.startswith("{")][-1])
    assert d5["steps"] == 5 and d5["gpu_launches"] == d["gpu_launches"] > 0, (d5["gpu_launches"], d["gpu_launches"])
