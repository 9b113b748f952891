"""Shared helpers for the test-suite (test infrastructure; may import the oracle)."""
import os

import numpy as np
import torch
from torch import nn

import stmgcn_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-4          # BASELINE.json north_star: "within 1e-4 relative fp32" (max-norm form, SURVEY 8(d))


def load_golden(name):
    """A fixture of oracle/make_golden.py: ``<name>.npz``, continued in ``<name>.1.npz``, ... when it is too large for
    one file.  Returns the meta dict, parameters, gradients, supports, adjacencies and a dict of every stored array."""
    paths = [os.path.join(GOLDEN, name + ".npz")]
    while os.path.exists(os.path.join(GOLDEN, f"{name}.{len(paths)}.npz")):
        paths.append(os.path.join(GOLDEN, f"{name}.{len(paths)}.npz"))
    blob = {}
    for path in paths:
        with np.load(path) as part:
            blob.update((key, part[key]) for key in part.files)
    n, m, k, t, b, c, hid, layers, gcn_hid = [int(v) for v in blob["meta"]]
    meta = dict(n=n, m=m, k=k, t=t, b=b, c=c, hid=hid, layers=layers, gcn_hid=gcn_hid)
    params = {key[len("param."):]: torch.from_numpy(blob[key]) for key in blob if key.startswith("param.")}
    grads = {key[len("grad."):]: blob[key] for key in blob if key.startswith("grad.")}
    supports = [torch.from_numpy(blob[f"supports.{g}"]) for g in range(m)]
    adjs = [torch.from_numpy(blob[f"adj.{g}"]) for g in range(m)]
    return meta, params, grads, supports, adjs, blob


def build_model(meta, device, relu=True):
    import STMGCN
    model = STMGCN.ST_MGCN(M=meta["m"], seq_len=meta["t"], n_nodes=meta["n"], input_dim=meta["c"],
                           lstm_hidden_dim=meta["hid"], lstm_num_layers=meta["layers"],
                           gcn_hidden_dim=meta["gcn_hid"],
                           sta_kernel_config={"kernel_type": "chebyshev", "K": meta["k"]},
                           gconv_use_bias=True, gconv_activation=nn.ReLU if relu else None)
    return model.to(device)


def assert_close(new, ref, what, tol=TOL):
    err = O.max_rel_err(new, ref)
    assert err <= tol, f"{what}: max-norm relative error {err:.3e} > {tol:.1e}"
    return err
