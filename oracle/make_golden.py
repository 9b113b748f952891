"""Generate ``tests/golden/*.npz`` by running the UNMODIFIED reference on CPU fp32.

TEST INFRASTRUCTURE.  Needs the original project staged under ``oracle/_ref/`` (``oracle/stage_reference.py``):

    python oracle/make_golden.py [case ...]          (default: every case)

Each fixture stores: the adjacency matrices, the reference's supports ``Adj_Preprocessor.process``
(``GCN.py:57-97``), the reference model's ``state_dict`` after ``torch.manual_seed(seed)`` construction,
inputs ``x, y``, the forward output of ``ST_MGCN.forward`` (``STMGCN.py:100-119``), the MSE loss and the
autograd gradient of every parameter.  Reference modules are imported under their own names from a
temporary ``sys.path`` entry and removed again so they can never shadow the repo's drop-in modules.
"""
from __future__ import annotations

import glob
import os
import sys

import numpy as np
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
REF = os.path.join(HERE, "_ref")            # oracle/stage_reference.py
GOLDEN = os.path.join(REPO, "tests", "golden")
PART_BYTES = 900_000


def import_reference():
    """Import the reference ``GCN`` / ``STMGCN`` modules as private objects (not left in sys.modules)."""
    if not os.path.exists(os.path.join(REF, "STMGCN.py")):
        raise FileNotFoundError(f"{REF} holds no staged reference: run oracle/stage_reference.py first")
    saved = {k: sys.modules.pop(k) for k in ("GCN", "STMGCN") if k in sys.modules}
    sys.path.insert(0, REF)
    try:
        import GCN as ref_gcn          # noqa: N811
        import STMGCN as ref_stmgcn    # noqa: N811
    finally:
        sys.path.remove(REF)
        for k in ("GCN", "STMGCN"):
            sys.modules.pop(k, None)
        sys.modules.update(saved)
    return ref_gcn, ref_stmgcn


def build_case(name, n, m, k, t, b, c, hid, layers, gcn_hid, density, seed, weighted=False):
    sys.path.insert(0, os.path.join(REPO, "st-mgcn_b200"))
    from stmgcn_b200 import synth
    ref_gcn, ref_stmgcn = import_reference()
    adjs = [synth.make_adjacency(n, g, density) for g in range(m)]
    if weighted:                                    # asymmetric, weighted => asymmetric L~
        gen = torch.Generator().manual_seed(77)
        adjs = [a * (0.25 + torch.rand(n, n, generator=gen)) for a in adjs]
    sups = [ref_gcn.Adj_Preprocessor("chebyshev", k).process(a) for a in adjs]
    torch.manual_seed(seed)
    model = ref_stmgcn.ST_MGCN(M=m, seq_len=t, n_nodes=n, input_dim=c, lstm_hidden_dim=hid,
                               lstm_num_layers=layers, gcn_hidden_dim=gcn_hid,
                               sta_kernel_config={"kernel_type": "chebyshev", "K": k},
                               gconv_use_bias=True, gconv_activation=nn.ReLU)
    x = torch.randn(b, t, n, c)
    y = torch.randn(b, n, c)
    out = model(obs_seq=x, sta_adj_list=sups)
    loss = nn.MSELoss(reduction="mean")(out, y)
    loss.backward()
    blob = {"meta": np.array([n, m, k, t, b, c, hid, layers, gcn_hid], dtype=np.int64),
            "x": x.numpy(), "y": y.numpy(), "out": out.detach().numpy(),
            "loss": np.array(loss.item(), dtype=np.float64)}
    for g, (a, s) in enumerate(zip(adjs, sups)):
        blob[f"adj.{g}"] = a.numpy()
        blob[f"supports.{g}"] = s.numpy()
    for key, val in model.state_dict().items():
        blob["param." + key] = val.numpy()
    for key, val in model.named_parameters():
        blob["grad." + key] = val.grad.numpy()
    paths = save_parts(name, blob)
    print(f"{name}: out|max|={float(out.abs().max()):.4g} loss={loss.item():.6f} -> "
          + ", ".join(f"{os.path.basename(p)} ({os.path.getsize(p) / 1024:.0f} KiB)" for p in paths))


def save_parts(name, blob):
    """Write ``tests/golden/<name>.npz``, continued in ``<name>.1.npz``, ``<name>.2.npz``, ... so that no file holds
    more than PART_BYTES of arrays (every fixture file stays under 1 MB; random weights do not compress).  Arrays keep
    their order across the parts; ``tests/helpers.load_golden`` merges them."""
    parts, size = [{}], 0
    for key, val in blob.items():
        if parts[-1] and size + val.nbytes > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][key] = val
        size += val.nbytes
    for stale in glob.glob(os.path.join(GOLDEN, name + ".[0-9]*.npz")):
        os.remove(stale)
    paths = [os.path.join(GOLDEN, name + (f".{i}" if i else "") + ".npz") for i in range(len(parts))]
    for path, part in zip(paths, parts):
        np.savez_compressed(path, **part)
        assert os.path.getsize(path) < 1_000_000, path
    return paths


CASES = {
    # BASELINE.json configs[0]: 64 regions, 1 graph, K=2, seq_len=4, batch=8, H=G=64, L=3, C=1.
    "cfg1_ref": dict(n=64, m=1, k=2, t=4, b=8, c=1, hid=64, layers=3, gcn_hid=64, density=0.10, seed=0),
    # ragged/small case: 3 graphs, weighted asymmetric adjacency, C=2, odd sizes.
    "ragged_ref": dict(n=37, m=3, k=3, t=5, b=3, c=2, hid=16, layers=2, gcn_hid=24, density=0.15, seed=1, weighted=True),
    # BASELINE.json configs[1]/[2] hyper-parameters (3 graphs, K=3, seq_len=12, H=G=64, L=3, C=1) at a size the reference
    # finishes in seconds: 96 regions x batch 6 = 576 LSTM rows (4.5 tiles of 128: ragged last tile on the GPU).
    "cfg3_small_ref": dict(n=96, m=3, k=3, t=12, b=6, c=1, hid=64, layers=3, gcn_hid=64, density=0.05, seed=2),
    # the dense restatement's own check (tests/test_oracle.py::test_dense_matches_reference_modules): 2 graphs, K=3,
    # H=16, L=2, G=8 -- small enough to keep every value
    "dense_check_ref": dict(n=30, m=2, k=3, t=5, b=2, c=1, hid=16, layers=2, gcn_hid=8, density=0.2, seed=3),
}


if __name__ == "__main__":
    torch.set_num_threads(1)
    for name in sys.argv[1:] or CASES:
        build_case(name, **CASES[name])
