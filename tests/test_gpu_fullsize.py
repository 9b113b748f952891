"""GPU parity at the sizes that are BENCHMARKED (BASELINE.json configs[1..4]), not only at toy sizes.

Windows of a batch are independent (``STMGCN.py:47``: every (window, region) pair is its own LSTM row; the only
reductions are over regions inside one window, ``STMGCN.py:42``, and over graphs, ``STMGCN.py:116``), so the fp64 sparse
oracle evaluated on a FEW windows pins the full-batch GPU run:

* forward: ``out[b]`` of the full-batch run must equal the oracle's output for window ``b``;
* backward: the targets of all other windows are set to the GPU's own forward output, so their residual -- and with it
  their gradient contribution -- vanishes; the full-batch gradient is then exactly ``|picked| / B`` times the oracle's
  gradient on the picked windows.  Every kernel still runs at the full size (262 144 LSTM rows, 2 048 tiles, > 2^31
  element tapes at cfg3), with the rows of the other windows carrying zeros through the backward.

Tolerance: 1e-4 max-norm relative (BASELINE.json north_star), fp32 arithmetic.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch
from torch import nn

import stmgcn_oracle as O
from helpers import TOL, assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _csr_of(sup):
    """scipy CSR of L~ from a ChebSupports handle (CPU copy)."""
    rp, ci, va = sup.rowptr.cpu().numpy(), sup.colidx.cpu().numpy(), sup.vals.cpu().numpy()
    return sp.csr_matrix((va, ci, rp), shape=(sup.n, sup.n))


def _build(w, batch, seed_x=100, relu=True):
    import GCN
    import STMGCN
    from stmgcn_b200 import synth
    pre = GCN.Adj_Preprocessor("chebyshev", w.cheb_order)
    sups_cpu = [pre.process_sparse(a) for a in synth.make_adjacency_list(w)]
    torch.manual_seed(0)
    kw = synth.model_kwargs(w)
    if not relu:
        kw["gconv_activation"] = None
    model = STMGCN.ST_MGCN(**kw)
    params = {k: v.detach().clone().numpy() for k, v in model.state_dict().items()}
    x, y = synth.make_inputs(w, seed=seed_x, batch=batch)
    return model.to(DEV), [s.to(DEV) for s in sups_cpu], [_csr_of(s) for s in sups_cpu], params, x, y


class _KinkAwareOracle(O.SparseOracle):
    """SparseOracle that records, per GCN call, how close the closest pre-activation is to the ReLU kink."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.kink = []                          # per _gcn_fwd call (order: temporal m0, spatial m0, temporal m1, ...)

    def _gcn_fwd(self, lap, x, w, b):
        s = self._cheb_stack(lap, x)
        p = x.shape[-1]
        z = sum(s[k] @ w[k * p:(k + 1) * p] for k in range(self.ks))
        if b is not None:
            z = z + b
        self.kink.append(float(np.min(np.abs(z)) / max(float(np.max(np.abs(z))), 1e-30)))
        return (np.maximum(z, 0) if self.relu else z), s


def _check_subbatch(w, batch, picks, tol=TOL, relu=True):
    """ReLU note.  With only a few windows carrying gradient, ONE pre-activation of a GCN that lands within rounding
    distance of zero flips its ReLU mask between fp32 and fp64 and moves every gradient of that graph branch by ~1e-3
    (one element out of ~10^6 active ones; measured: the same flip appears with the first- and the second-generation
    kernels on different inputs, never in a full batch).  The fp32 reference itself has the same property.  So the ReLU
    variant checks forward + loss strictly and the gradients of a branch strictly only when the oracle finds no
    pre-activation closer than 1e-5 (relative) to the kink; the variant without activation (smooth) checks everything."""
    model, sups, laps, params, x, y = _build(w, batch, relu=relu)
    crit = nn.MSELoss(reduction="mean")
    xd = x.to(DEV)
    with torch.no_grad():
        out0 = model(obs_seq=xd, sta_adj_list=sups)
    # targets: the run's own output everywhere except the picked windows
    y2 = out0.detach().clone()
    y2[picks] = y[picks].to(DEV)
    out = model(obs_seq=xd, sta_adj_list=sups)
    loss = crit(out, y2)
    loss.backward()
    torch.cuda.synchronize()
    orc = _KinkAwareOracle(params, laps, w.n_supports, relu=relu, dtype=np.float64)
    o_ref, l_ref, g_ref = orc.loss_and_grads(x[picks].numpy(), y[picks].numpy())
    scale = len(picks) / float(batch)
    errs = {"out": O.max_rel_err(out.detach()[picks].cpu().numpy(), o_ref),
            "loss": abs(loss.item() - l_ref * scale) / abs(l_ref * scale)}
    for key, p in model.named_parameters():
        errs["grad " + key] = O.max_rel_err(p.grad.cpu().numpy(), g_ref[key] * scale)
    # a branch is "near a kink" if any of its two GCNs has a pre-activation within 1e-5 of zero (relative to max |z|)
    near = [relu and min(orc.kink[2 * m], orc.kink[2 * m + 1]) < 1e-5 for m in range(w.n_graphs)]
    print(f"{w.name} B={batch} relu={relu} windows {picks}: kink distance per branch "
          f"{[f'{min(orc.kink[2 * m], orc.kink[2 * m + 1]):.1e}' for m in range(w.n_graphs)]}; max-norm relative errors vs "
          f"the fp64 oracle: " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(errs.items(), key=lambda kv: -kv[1])[:6]))

    def tol_of(key):
        for m in range(w.n_graphs):
            if near[m] and (f"rnn_list.{m}." in key or f"gcn_list.{m}." in key):
                return 5e-2
        return tol
    bad = {k: v for k, v in errs.items() if not (v <= tol_of(k))}
    assert not bad, f"{w.name} B={batch}: above tolerance: {bad}"
    assert bool(torch.isfinite(out).all())                  # every window, not only the picked ones
    return errs


@pytest.mark.parametrize("relu", [True, False])
def test_cfg3_full_size_vs_fp64_oracle_on_two_windows(relu):
    """BASELINE configs[2]: 4096 regions, 3 graphs, K=3, T=12, batch 64, fp32 -- the size bench.py reports."""
    from stmgcn_b200 import synth
    _check_subbatch(synth.WORKLOADS["cfg3"], 64, [0, 63], relu=relu)


@pytest.mark.parametrize("relu", [True, False])
def test_cfg2_full_size_vs_fp64_oracle(relu):
    """BASELINE configs[1] shapes (1024 regions, 3 graphs, K=3, T=12, batch 32) in fp32 against the oracle on 3 windows."""
    from stmgcn_b200 import synth
    _check_subbatch(synth.WORKLOADS["cfg2"], 32, [0, 17, 31], relu=relu)


@pytest.mark.parametrize("relu", [True, False])
def test_cfg5_shapes_vs_fp64_oracle_on_one_window(relu):
    """BASELINE configs[4] shapes: 16384 regions, 3 graphs at 1 % density, K=5 (six supports), T=24; batch 8 of 32."""
    from stmgcn_b200 import synth
    _check_subbatch(synth.WORKLOADS["cfg5"], 8, [5], relu=relu)


def test_lstm_tensor_core_vs_exact_fp32_at_cfg3_size():
    """tcgen05 LSTM forward + BPTT + weight gradients against the exact-FFMA kernels ON DEVICE at cfg3's 262 144 rows."""
    from stmgcn_b200 import ops
    n, b, t, hid, lyr = 4096, 64, 12, 64, 3
    gen = torch.Generator().manual_seed(5)
    xo = torch.randn(n, b, t, 1, generator=gen).to(DEV)
    s0 = torch.rand(b, t, generator=gen).to(DEV)
    ws0 = []
    for l in range(lyr):
        in_l = 1 if l == 0 else hid
        ws0 += [(torch.rand(4 * hid, in_l, generator=gen) - 0.5) * 0.25, (torch.rand(4 * hid, hid, generator=gen) - 0.5) * 0.25,
                (torch.rand(4 * hid, generator=gen) - 0.5) * 0.25, (torch.rand(4 * hid, generator=gen) - 0.5) * 0.25]
    proj = (torch.randn(n, b, hid, generator=gen) * 1e-3).to(DEV)
    res = {}
    old = ops.lstm_path()
    try:
        for path in ("fma", "tc"):
            ops.set_lstm_path(path)
            s = s0.clone().requires_grad_(True)
            ws = [w_.to(DEV).requires_grad_(True) for w_ in ws0]
            h_top, _, _ = ops.SharedLSTM.apply(xo, s, None, None, lyr, hid, False, *ws)
            (h_top * proj).sum().backward()
            res[path] = [h_top.detach().clone(), s.grad.clone()] + [w_.grad.clone() for w_ in ws]
            del h_top, s, ws
            torch.cuda.empty_cache()
    finally:
        ops.set_lstm_path(old)
    names = ["h_top", "d_s"] + [f"w{i}" for i in range(4 * lyr)]
    # weight gradients are sums over 3.1 M (row, step) pairs: the two kernels add them in different orders in fp32, which
    # alone is worth ~1e-4 relative (measured 9.4e-5 between the first-generation 3xTF32 LSTM kernels and the FFMA
    # kernels); the fp64-oracle tests above are the pin, this one guards against indexing bugs at > 2^31-element sizes
    for name, a, c in zip(names, res["tc"], res["fma"]):
        assert_close(a.cpu().numpy(), c.cpu().numpy(), f"cfg3-size tc vs fma {name}", 5e-5 if name in ("h_top",) else 3e-4)


def test_cg_lstm_and_model_with_localpool_supports():
    """kernel_type='localpool' (A[0] = I + A_norm != I): the context gate's residual is x itself, not A_0 x
    (STMGCN.py:40-41).  CG_LSTM and ST_MGCN forward + every gradient against the dense oracle."""
    import GCN
    import STMGCN
    from stmgcn_b200 import synth
    n, b, t, c, hid, lyr, gh, m = 60, 5, 6, 1, 64, 2, 24, 2
    pre = GCN.Adj_Preprocessor("localpool", 1)
    sups = [pre.process(synth.make_adjacency(n, g, 0.15)) for g in range(m)]
    torch.manual_seed(3)
    model = STMGCN.ST_MGCN(M=m, seq_len=t, n_nodes=n, input_dim=c, lstm_hidden_dim=hid, lstm_num_layers=lyr,
                           gcn_hidden_dim=gh, sta_kernel_config={"kernel_type": "localpool", "K": 1},
                           gconv_use_bias=True, gconv_activation=nn.ReLU)
    params = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(DEV)
    gen = torch.Generator().manual_seed(9)
    x, y = torch.randn(b, t, n, c, generator=gen), torch.randn(b, n, c, generator=gen)
    out = model(obs_seq=x.to(DEV), sta_adj_list=[s.to(DEV) for s in sups])
    loss = nn.MSELoss()(out, y.to(DEV))
    loss.backward()
    ref_p = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    ref_out = O.dense_st_mgcn(ref_p, x, sups)
    ref_loss = nn.MSELoss()(ref_out, y)
    ref_loss.backward()
    assert_close(out.detach().cpu().numpy(), ref_out.detach().numpy(), "localpool model forward")
    for key, p in model.named_parameters():
        assert_close(p.grad.cpu().numpy(), ref_p[key].grad.numpy(), f"localpool grad {key}")
    # CG_LSTM alone (the advisor's case): gate computed from x + gconv(x)
    cg = model.rnn_list[0]
    h0 = cg.init_hidden(b)
    o1, _ = cg(sups[0].to(DEV), x.to(DEV), h0)
    o_ref, _ = O.dense_cg_lstm(sups[0], x, {"p." + k[len("rnn_list.0."):]: v for k, v in params.items()
                                             if k.startswith("rnn_list.0.")}, "p.")
    assert_close(o1.detach().cpu().numpy(), o_ref.numpy(), "localpool CG_LSTM forward")
