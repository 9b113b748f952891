"""Drop-in: the reference's OWN ``Main.py`` / ``Model_Trainer.py`` / ``Data_Container.py`` run UNCHANGED on this repo's
``GCN`` / ``STMGCN`` modules (BASELINE.json north_star: "Main.py and Model_Trainer.py run unchanged"; SURVEY.md section 4
"drop-in" row, section 8(c) bullet 2).

The five reference files are staged, byte for byte, under the git-ignored ``oracle/_ref/`` by
``oracle/stage_reference.py`` (``__graft_entry__.build()`` runs it when it finds a checkout of the original) and
checked against their SHA-256 in ``tests/golden/reference_sha256.json``.  The original sources are not part of this
repository, so the test skips where nothing was staged.  The script is driven through its own command line only
(``--device``, ``--dates``): nothing is patched, the hard-coded ``epoch = 100`` (``Main.py:11``) runs with the
trainer's own early stopping (``Model_Trainer.py:54-60``) on a synthetic ``./data/data_dict.npz`` (the dataset is not
shipped, ``Main.py:9``): ``taxi (T,58,1)`` plus three ``(58,58)`` adjacencies.
"""
import hashlib
import io
import json
import os
import re
import runpy
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(REPO, "oracle", "_ref")


def _write_dataset(path, hours=24 * 16, n=58, seed=0):
    rng = np.random.default_rng(seed)
    t = np.arange(hours)[:, None, None]
    base = 20 + 10 * np.sin(2 * np.pi * t / 24.0 + rng.uniform(0, 6.28, (1, n, 1)))      # daily rhythm per region
    taxi = np.maximum(base + rng.normal(0, 2.0, (hours, n, 1)), 0).astype(np.float64)
    blob = {"taxi": taxi}
    for key, dens in (("neighbor_adj", 0.08), ("trans_adj", 0.12), ("semantic_adj", 0.2)):
        a = (rng.random((n, n)) < dens).astype(np.float64)
        a = np.maximum(a, a.T)
        np.fill_diagonal(a, 0)
        idx = np.arange(n)
        a[idx, (idx + 1) % n] = a[(idx + 1) % n, idx] = 1          # no isolated region (GCN.py:109 would emit NaN)
        blob[key] = a
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez(path, **blob)


@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "Main.py")),
                    reason="original project not staged (build() stages it from a checkout it finds, or run "
                           "python oracle/stage_reference.py <its checkout>)")
def test_reference_main_runs_unchanged_on_the_b200_modules(tmp_path):
    from stmgcn_b200 import _lib
    # the staged files are the unmodified original (SHA-256 of commit 5ee7e17): the test must not run a doctored script
    with open(os.path.join(REPO, "tests", "golden", "reference_sha256.json")) as fh:
        digests = json.load(fh)
    for name, digest in digests.items():
        with open(os.path.join(REF, name), "rb") as fh:
            assert hashlib.sha256(fh.read()).hexdigest() == digest, f"oracle/_ref/{name} differs from the original"
    _write_dataset(str(tmp_path / "data" / "data_dict.npz"))
    saved_path, saved_argv, saved_cwd = list(sys.path), list(sys.argv), os.getcwd()
    saved_mods = {k: sys.modules.pop(k) for k in ("GCN", "STMGCN", "Model_Trainer", "Data_Container") if k in sys.modules}
    launches0 = _lib.launch_count()
    buf = io.StringIO()
    try:
        os.chdir(tmp_path)
        # INTEGRATION.md section 1: this repo first (its GCN.py / STMGCN.py win `import GCN, STMGCN`, Main.py:5),
        # then the reference directory (Data_Container, Model_Trainer)
        sys.path[:0] = [REPO, os.path.join(REPO, "st-mgcn_b200"), REF]
        # train on one week of hourly windows (135 train -> last batch of 7, 33 validate), test on two days
        sys.argv = ["Main.py", "--device", "cuda:0", "--dates", "0101", "0107", "0108", "0109"]
        torch.manual_seed(1234)        # Main.py sets no seed: fix the parameter init so the run is comparable (see below)
        with redirect_stdout(buf):
            runpy.run_path(os.path.join(REF, "Main.py"), run_name="__main__")
        used = {k: os.path.abspath(sys.modules[k].__file__) for k in ("GCN", "STMGCN", "Model_Trainer", "Data_Container")}
    finally:
        os.chdir(saved_cwd)
        sys.path[:] = saved_path
        sys.argv[:] = saved_argv
        for k in ("GCN", "STMGCN", "Model_Trainer", "Data_Container"):
            sys.modules.pop(k, None)
        sys.modules.update(saved_mods)
    log = buf.getvalue()
    # our modules were the ones imported, the trainer / data code was the reference's
    assert used["GCN"] == os.path.join(REPO, "GCN.py") and used["STMGCN"] == os.path.join(REPO, "STMGCN.py"), used
    assert used["Model_Trainer"] == os.path.join(REF, "Model_Trainer.py"), used
    assert used["Data_Container"] == os.path.join(REF, "Data_Container.py"), used
    assert _lib.launch_count() - launches0 > 1000, "the run did not go through libstmgcn_b200.so"
    # it trained, checkpointed, reloaded and printed the reference's metrics (Model_Trainer.py:47-63, :68-98)
    assert "Training starts at" in log and "Update model checkpoint" in log and "Testing ends at" in log, log[-2000:]
    for metric in ("test true MSE", "test true RMSE", "test true MAE", "test true MAPE"):
        assert metric in log, log[-2000:]
    rmse = float(log.split("test true RMSE:")[1].split()[0])
    drops = [float(v) for v in re.findall(r"to ([0-9.eE+-]+)\. Update model checkpoint", log)]
    # anchors: the UNMODIFIED reference (its own GCN/STMGCN on the CPU, same script, same synthetic file, same
    # torch.manual_seed(1234)) printed these validation losses for epochs 1-3 and "test true RMSE: 2.31858" in the build
    # container.  Same seed => bit-identical init here (tests/test_abi_and_host.py), so the first epochs (15 Adam steps)
    # must track the reference closely; 100 epochs later only the converged error is comparable.
    ref_first, ref_rmse = [0.19774, 0.19067, 0.16364], 2.31858
    assert len(drops) >= 3, drops
    for got, want in zip(drops[:3], ref_first):
        assert abs(got - want) / want < 0.02, (drops[:3], ref_first)
    assert drops[-1] < 0.25 * drops[0], drops
    assert np.isfinite(rmse) and abs(rmse - ref_rmse) / ref_rmse < 0.10, rmse
    ckpt = torch.load(tmp_path / "output" / "ST_MGCN_best_model.pkl", map_location="cpu")
    keys = set(ckpt["state_dict"].keys())
    assert "rnn_list.0.lstm.weight_ih_l0" in keys and "gcn_list.2.W" in keys and "fc.weight" in keys
    print(log[-1200:])
