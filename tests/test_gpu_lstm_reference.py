"""Both shared-LSTM kernel families against an fp64 LSTM, at every edge of their whole-sequence schedule.

The op under test is ``ops.SharedLSTM``: rows r = n*B + b, input ``xo[n, b, t, :] * s[b, t]``, optional initial state
(h0, c0).  The reference is ``O.lstm_explicit`` in float64 on the CPU with autograd (pinned to ``nn.LSTM`` in
``test_oracle.py``; the row order and gate scaling of this file's own helper are pinned by the CPU test at the bottom).
Every case compares h_top, h_n, c_n, d_s and all 4*L weight gradients under the loss ``sum(h_top * proj)``, and asserts
which kernel family ran, so a routing change cannot silently change what a case tests.

Schedule edges of the tensor-core family (lstm16.cu), one named case each:
* L = 1 (no dx_work), L = 2 (one dx_work slice), L >= 4 (slices reused), L = 8 (the limit), with and without (h0, c0):
  the backward reads h0 at t = 0 (and c0 as c_prev) only with an initial state;
* C = 1 (the one-channel kernel variant) and C = 2, 3, 4 (the runtime-channel variant, layer-0 W_ih gradient);
* rows 1, 127, 128, 129 and a ragged multi-tile size;
* T = 1, 56 and 64 (the backward's limit).  At one tile per CTA a launch covers up to 48 steps, so T = 56 runs as
  48 + 8 and T = 64 as 48 + 16: a short last launch, weight gradients accumulated across launches, dh_rec / dc carried;
* d_s through global atomics in one launch and shared memory in the next (steps * B > 1024, then <= 1024);
* several tiles per CTA, with a short last launch (test_tensor_core_family_several_tiles_per_cta_short_last_launch).
"""
import math

import numpy as np
import pytest
import torch

import stmgcn_oracle as O
from helpers import assert_close

DEV = "cuda:0"
TC, EXACT = "SharedLSTM16Backward", "SharedLSTMExactBackward"
TOL_TC = 1e-4           # 3xBF16 planes, the project's fp32 parity bar
TOL_EXACT = 1e-5        # fp32 FFMA against fp64
TOL_BF16 = 2e-2         # single-pass bf16 (planes = 1): the bar of test_bf16_arithmetic_mode_within_the_reference_bf16_tolerance
NAMES = ("h_top", "h_n", "c_n", "d_s")


# --------------------------------------------------------------------------------------------------
# inputs and the fp64 reference
# --------------------------------------------------------------------------------------------------
def _make_case(n, b, t, c, n_layers, hid, state, seed):
    """fp32 CPU tensors: xo (N,B,T,C), s (B,T), h0 / c0 (L, N*B, H) or None, nn.LSTM weights from U(-0.25, 0.25)
    (the gates stay away from saturation), proj (N,B,H)."""
    gen = torch.Generator().manual_seed(seed)

    def uni(*shape, bound=0.25):
        return (torch.rand(*shape, generator=gen) * 2 - 1) * bound

    xo = torch.randn(n, b, t, c, generator=gen)
    s = torch.rand(b, t, generator=gen)
    weights = []
    for l in range(n_layers):
        in_l = c if l == 0 else hid
        weights += [uni(4 * hid, in_l), uni(4 * hid, hid), uni(4 * hid), uni(4 * hid)]
    h0 = uni(n_layers, n * b, hid, bound=0.5) if state else None
    c0 = uni(n_layers, n * b, hid, bound=1.0) if state else None
    proj = torch.randn(n, b, hid, generator=gen)
    return xo, s, h0, c0, weights, proj


def _fp64_reference(xo, s, h0, c0, weights, proj, rows=None):
    """fp64 autograd through ``O.lstm_explicit`` of the shared LSTM on rows r = n*B + b (all of them, or the index
    tensor ``rows``), input ``xo[n, b, t, :] * s[b, t]``, constant (h0, c0), loss ``sum(h_top * proj[rows])``.
    Windows are independent, so on a subset of rows this is the full run's result on those rows, and its d_s and
    weight gradients equal the full run's when ``proj`` is zero on every other row."""
    n, b, t_len, c_in = xo.shape
    n_layers = len(weights) // 4
    s = s.detach().double().clone().requires_grad_(True)
    ws = [w.detach().double().clone().requires_grad_(True) for w in weights]
    x = (xo.double() * s[None, :, :, None]).reshape(n * b, t_len, c_in)
    p = proj.double().reshape(n * b, -1)
    if rows is not None:
        x, p = x[rows], p[rows]
        h0 = h0[:, rows] if h0 is not None else None
        c0 = c0[:, rows] if c0 is not None else None
    h0 = h0.double() if h0 is not None else None
    c0 = c0.double() if c0 is not None else None
    seq, (h_n, c_n) = O.lstm_explicit(x, [tuple(ws[4 * l:4 * l + 4]) for l in range(n_layers)], h0, c0)
    h_top = seq[:, -1]
    loss = (h_top * p).sum()
    loss.backward()
    return dict(h_top=h_top.detach(), h_n=h_n.detach(), c_n=c_n.detach(), d_s=s.grad, grads=[w.grad for w in ws],
                loss=loss.item())


def _run_device(xo, s, h0, c0, weights, proj, hid):
    """ops.SharedLSTM forward (want_state=True) + backward of ``sum(h_top * proj)`` on the GPU."""
    from stmgcn_b200 import ops
    n, b = xo.shape[:2]
    n_layers = len(weights) // 4
    s_d = s.to(DEV).requires_grad_(True)
    ws = [w.to(DEV).requires_grad_(True) for w in weights]
    h_top, h_n, c_n = ops.SharedLSTM.apply(xo.to(DEV), s_d, h0.to(DEV) if h0 is not None else None,
                                           c0.to(DEV) if c0 is not None else None, n_layers, hid, True, *ws)
    family = type(h_top.grad_fn).__name__
    (h_top * proj.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    return family, dict(h_top=h_top.detach().reshape(n * b, hid).cpu(), h_n=h_n.cpu(), c_n=c_n.cpu(), d_s=s_d.grad.cpu(),
                        grads=[w.grad.cpu() for w in ws])


def _errors(got, ref, rows=None):
    """max-norm relative error of every compared quantity: h_top, h_n, c_n (on ``rows``), d_s, w0 .. w{4L-1}."""
    pick = (lambda v: v) if rows is None else (lambda v: v[..., rows, :])
    errs = {"h_top": O.max_rel_err(pick(got["h_top"]).numpy(), ref["h_top"].numpy())}
    for key in ("h_n", "c_n"):
        errs[key] = O.max_rel_err(pick(got[key]).numpy(), ref[key].numpy())
    errs["d_s"] = O.max_rel_err(got["d_s"].numpy(), ref["d_s"].numpy())
    for i, (g, r) in enumerate(zip(got["grads"], ref["grads"])):
        errs[f"w{i}"] = O.max_rel_err(g.numpy(), r.numpy())
    return errs


def _report(name, family, errs):
    worst = max(errs, key=errs.get)
    print(f"[lstm vs fp64] {name}: {family}, worst max-norm relative error {errs[worst]:.2e} ({worst})")


def _check(name, errs, tol):
    bad = {k: f"{v:.2e}" for k, v in errs.items() if not v <= tol}
    assert not bad, f"{name}: above {tol:.0e} against fp64: {bad}"


def _run_case(name, n, b, t, c, n_layers, hid, state, family, tol, seed=0):
    xo, s, h0, c0, weights, proj = _make_case(n, b, t, c, n_layers, hid, state, seed)
    got_family, got = _run_device(xo, s, h0, c0, weights, proj, hid)
    assert got_family == family, f"{name}: ran {got_family}, the case is there to test {family}"
    errs = _errors(got, _fp64_reference(xo, s, h0, c0, weights, proj))
    _report(name, got_family, errs)
    _check(name, errs, tol)
    return errs


@pytest.fixture
def lstm_mode():
    """ops with its kernel-family switches restored after the test."""
    from stmgcn_b200 import ops
    old = ops.lstm_path(), ops.lstm_planes()
    yield ops
    ops.set_lstm_path(old[0])
    ops.set_lstm_planes(old[1])


# --------------------------------------------------------------------------------------------------
# tensor-core family (lstm16.cu), 3xBF16 planes
# --------------------------------------------------------------------------------------------------
# name: (N, B, T, C, L, initial state)
TC_CASES = {
    "rows1_T1_L1": (1, 1, 1, 1, 1, False),
    "rows1_T1_L1_state": (1, 1, 1, 1, 1, True),
    "rows127_T5_C3_L2_state": (127, 1, 5, 3, 2, True),
    "rows128_T6_C4_L4": (32, 4, 6, 4, 4, False),
    "rows129_T4_C2_L8_state": (43, 3, 4, 2, 8, True),
    "rows130_T1_C1_L8": (10, 13, 1, 1, 8, False),
    "rows333_ragged_T7_C1_L4_state": (37, 9, 7, 1, 4, True),
    "rows2200_ds_global_T3_C2_L2": (2, 1100, 3, 2, 2, False),
    # 48 + 8 steps: d_s through global atomics in the first launch (48 * 22 > 1024), shared memory in the second
    "T56_ds_global_then_shared_C3_L2_state": (3, 22, 56, 3, 2, True),
    "T56_48+8_C2_L1": (4, 16, 56, 2, 1, False),
    "T64_48+16_C4_L2_state": (5, 20, 64, 4, 2, True),
    "T64_48+16_C1_L4": (3, 30, 64, 1, 4, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TC_CASES))
def test_tensor_core_family_matches_fp64(name, lstm_mode):
    lstm_mode.set_lstm_path("tc")
    lstm_mode.set_lstm_planes(2)
    n, b, t, c, n_layers, state = TC_CASES[name]
    _run_case(name, n, b, t, c, n_layers, 64, state, TC, TOL_TC)


@pytest.mark.gpu
def test_tensor_core_family_several_tiles_per_cta_short_last_launch(lstm_mode):
    """rows = N*B spans 2*grid + 2 tiles (grid = one CTA per SM), the last one ragged: 3 tiles per CTA, so one backward
    launch covers 48 / 3 = 16 steps and T = 20 runs as 16 + 4 per layer.  proj is zero except on every row of tiles
    0, grid, 2*grid and the last tile, so the fp64 reference runs on those rows alone; all other rows carry exact zeros
    through the backward and add nothing to d_s or the weight gradients."""
    from stmgcn_b200 import _lib
    lstm_mode.set_lstm_path("tc")
    lstm_mode.set_lstm_planes(2)
    grid = int(_lib.lib.stmgcn_sm_count())
    b, t, c, n_layers, hid = 7, 20, 3, 2, 64
    n = ((2 * grid + 1) * 128) // b + 1                  # rows in ((2 grid + 1) * 128, (2 grid + 1) * 128 + b]
    rows_total = n * b
    n_tiles = math.ceil(rows_total / 128)
    assert rows_total % 128 != 0 and n_tiles == 2 * grid + 2 and int(_lib.lib.stmgcn_lstm16_grid(rows_total)) == grid
    xo, s, h0, c0, weights, _ = _make_case(n, b, t, c, n_layers, hid, True, seed=3)
    picked = torch.cat([torch.arange(tile * 128, min((tile + 1) * 128, rows_total))
                        for tile in (0, grid, 2 * grid, n_tiles - 1)])
    gen = torch.Generator().manual_seed(4)
    proj = torch.zeros(rows_total, hid)
    proj[picked] = torch.randn(len(picked), hid, generator=gen)
    proj = proj.reshape(n, b, hid)

    from stmgcn_b200 import ops
    s_d = s.to(DEV).requires_grad_(True)
    ws = [w.to(DEV).requires_grad_(True) for w in weights]
    h_top, h_n, c_n = ops.SharedLSTM.apply(xo.to(DEV), s_d, h0.to(DEV), c0.to(DEV), n_layers, hid, True, *ws)
    family = type(h_top.grad_fn).__name__
    assert family == TC
    torch.cuda.synchronize()
    before = _lib.launch_count()
    (h_top * proj.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    launches = _lib.launch_count() - before
    # one weight-gradient reduction per layer, the rest are the fused backward launches
    per_layer = (launches - n_layers) / n_layers
    assert per_layer >= 2, f"{launches} backward launches for {n_layers} layers: the case no longer splits a layer"
    got = dict(h_top=h_top.detach().reshape(rows_total, hid).cpu(), h_n=h_n.cpu(), c_n=c_n.cpu(), d_s=s_d.grad.cpu(),
               grads=[w.grad.cpu() for w in ws])
    errs = _errors(got, _fp64_reference(xo, s, h0, c0, weights, proj, rows=picked), rows=picked)
    name = f"rows{rows_total}_{n_tiles}tiles_grid{grid}_T20_{per_layer:.0f}launches_per_layer"
    _report(name, family, errs)
    _check(name, errs, TOL_TC)


# --------------------------------------------------------------------------------------------------
# exact-fp32 family (lstm.cu)
# --------------------------------------------------------------------------------------------------
# name: (N, B, T, C, L, H, initial state, lstm_path)
EXACT_CASES = {
    "H4_C1_L1": (3, 5, 4, 1, 1, 4, False, "tc"),
    "H4_C4_L2_state": (6, 7, 3, 4, 2, 4, True, "tc"),
    "H36_C3_L2_state": (7, 9, 5, 3, 2, 36, True, "tc"),
    "H36_C1_L8": (5, 4, 3, 1, 8, 36, False, "tc"),
    "H100_C4_L8_state": (6, 11, 3, 4, 8, 100, True, "tc"),
    "H128_C3_L1_state": (5, 6, 4, 3, 1, 128, True, "tc"),
    # B > 2048: d_s through global atomics
    "H128_C1_L2_B2049": (2, 2049, 3, 1, 2, 128, False, "tc"),
    "H36_C3_L2_B2049_state": (1, 2049, 2, 3, 2, 36, True, "tc"),
    "H64_fma_C3_L2_state": (9, 5, 6, 3, 2, 64, True, "fma"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EXACT_CASES))
def test_exact_family_matches_fp64(name, lstm_mode):
    n, b, t, c, n_layers, hid, state, path = EXACT_CASES[name]
    lstm_mode.set_lstm_path(path)
    _run_case(name, n, b, t, c, n_layers, hid, state, EXACT, TOL_EXACT)


# --------------------------------------------------------------------------------------------------
# routing and the single-pass bf16 mode
# --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("t,family,tol", [(64, TC, TOL_TC), (65, EXACT, TOL_EXACT)])
def test_routing_boundary_at_T64(t, family, tol, lstm_mode):
    """H = 64 on the tc path: the tensor-core backward covers T <= 64, so T = 65 is routed to the exact family."""
    lstm_mode.set_lstm_path("tc")
    lstm_mode.set_lstm_planes(2)
    _run_case(f"routing_T{t}", 4, 6, t, 2, 2, 64, True, family, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rows127_T5_C3_L2_state", "rows333_ragged_T7_C1_L4_state",
                                  "T56_ds_global_then_shared_C3_L2_state", "rows128_T6_C4_L4"])
def test_single_pass_bf16_within_its_tolerance(name, lstm_mode):
    """planes = 1 stores h as one bf16 plane and runs its products single-pass.  Every error must stay within the
    mode's bar and be above 1e-6: fp32-grade results would mean the single-pass path did not run."""
    lstm_mode.set_lstm_path("tc")
    lstm_mode.set_lstm_planes(1)
    n, b, t, c, n_layers, state = TC_CASES[name]
    errs = _run_case("planes1_" + name, n, b, t, c, n_layers, 64, state, TC, TOL_BF16)
    fp32_grade = {k: f"{v:.1e}" for k, v in errs.items() if not v > 1e-6}
    assert not fp32_grade, f"planes1_{name}: fp32-grade errors, the single-pass path did not run: {fp32_grade}"


# --------------------------------------------------------------------------------------------------
# the public route to the initial-state backward: training a standalone CG_LSTM
# --------------------------------------------------------------------------------------------------
def _family_in_graph(t):
    """Names of the SharedLSTM autograd nodes reachable from ``t.grad_fn``."""
    seen, todo, found = set(), [t.grad_fn], set()
    while todo:
        fn = todo.pop()
        if fn is None or fn in seen:
            continue
        seen.add(fn)
        if type(fn).__name__ in (TC, EXACT):
            found.add(type(fn).__name__)
        todo += [nxt for nxt, _ in fn.next_functions]
    return found


@pytest.mark.gpu
@pytest.mark.parametrize("hid,family", [(64, TC), (36, EXACT)])
@pytest.mark.parametrize("hidden", ["init_hidden", "random"])
def test_cg_lstm_training_step_with_hidden_matches_fp64(hid, family, hidden, lstm_mode):
    """CG_LSTM.forward always hands ``hidden`` to the LSTM, and the zeros of ``init_hidden`` are a real tensor, so
    training a standalone CG_LSTM runs the initial-state backward.  Every parameter gradient (temporal GCN and fc
    through d_s, the LSTM directly) against ``O.dense_cg_lstm`` under fp64 autograd.  No GCN activation: with ReLU one
    temporal-GCN pre-activation near zero could flip between fp32 and fp64, which says nothing about the LSTM."""
    import STMGCN
    from stmgcn_b200 import synth
    lstm_mode.set_lstm_path("tc")
    lstm_mode.set_lstm_planes(2)
    n, b, t, c, n_layers, k = (40, 3, 6, 2, 2, 2) if hid == 64 else (30, 4, 5, 3, 3, 2)
    sup = O.chebyshev_supports_dense(synth.make_adjacency(n, 0, 0.2), k)
    torch.manual_seed(hid)
    mod = STMGCN.CG_LSTM(seq_len=t, n_nodes=n, input_dim=c, lstm_hidden_dim=hid, lstm_num_layers=n_layers, K=k + 1,
                         gconv_use_bias=True, gconv_activation=None).to(DEV)
    gen = torch.Generator().manual_seed(hid + 1)
    obs = torch.randn(b, t, n, c, generator=gen)
    proj = torch.randn(b, n, hid, generator=gen)
    if hidden == "init_hidden":
        h0, c0 = mod.init_hidden(b)
    else:
        h0 = ((torch.rand(n_layers, b * n, hid, generator=gen) * 2 - 1) * 0.5).to(DEV)
        c0 = (torch.rand(n_layers, b * n, hid, generator=gen) * 2 - 1).to(DEV)
    out, (h_n, c_n) = mod(sup.to(DEV), obs.to(DEV), (h0, c0))
    assert _family_in_graph(out) == {family}
    mod.zero_grad()
    (out * proj.to(DEV)).sum().backward()
    torch.cuda.synchronize()

    params = {"p." + key: v.detach().cpu().double().requires_grad_(True) for key, v in mod.named_parameters()}
    # the context gate's own ReLU (STMGCN.py:43) must not sit on its kink either
    fw, fb = params["p.fc.weight"].detach(), params["p.fc.bias"].detach()
    z = (obs.double().sum(-1).permute(0, 2, 1)
         + O.dense_gcn(sup.double(), obs.double().sum(-1).permute(0, 2, 1), params["p.gconv_temporal_feats.W"].detach(),
                       params["p.gconv_temporal_feats.b"].detach(), relu=False)).sum(1) / n
    a1 = z @ fw.t() + fb
    assert float(a1.abs().min() / a1.abs().max()) > 1e-4, "context-gate ReLU input within rounding of its kink"
    ref, (h_n_r, c_n_r) = O.dense_cg_lstm(sup.double(), obs.double(), params, "p.", relu=False,
                                           hidden=(h0.cpu().double(), c0.cpu().double()))
    (ref * proj.double()).sum().backward()
    errs = {"out": O.max_rel_err(out.detach().cpu().numpy(), ref.detach().numpy()),
            "h_n": O.max_rel_err(h_n.cpu().numpy(), h_n_r.detach().numpy()),
            "c_n": O.max_rel_err(c_n.cpu().numpy(), c_n_r.detach().numpy())}
    for key, p in mod.named_parameters():
        assert p.grad is not None, key
        errs["grad " + key] = O.max_rel_err(p.grad.cpu().numpy(), params["p." + key].grad.numpy())
    name = f"CG_LSTM_H{hid}_{hidden}"
    _report(name, family, errs)
    _check(name, errs, TOL_TC)


# --------------------------------------------------------------------------------------------------
# CPU: the reference helper itself
# --------------------------------------------------------------------------------------------------
def test_fp64_reference_row_order_and_gate_scaling():
    """The helper above, fed node-major rows n*B + b, agrees with ``nn.LSTM`` (``O.lstm_library``) fed ``obs * s`` in the
    reference's b*N + n row order (STMGCN.py:44, :47), and its d_s agrees with a central finite difference in s."""
    b, t, n, c, n_layers, hid = 2, 3, 4, 2, 2, 5
    gen = torch.Generator().manual_seed(0)
    obs = torch.randn(b, t, n, c, generator=gen, dtype=torch.float64)
    s = torch.rand(b, t, generator=gen, dtype=torch.float64) + 0.5
    weights = []
    for l in range(n_layers):
        in_l = c if l == 0 else hid
        weights += [(torch.rand(*shape, generator=gen, dtype=torch.float64) * 2 - 1) * 0.5
                    for shape in ((4 * hid, in_l), (4 * hid, hid), (4 * hid,), (4 * hid,))]
    h0_ref = torch.randn(n_layers, b * n, hid, generator=gen, dtype=torch.float64) * 0.5     # rows b*N + n
    c0_ref = torch.randn(n_layers, b * n, hid, generator=gen, dtype=torch.float64) * 0.5
    proj = torch.randn(n, b, hid, generator=gen, dtype=torch.float64)

    to_node_major = lambda v: v.reshape(n_layers, b, n, hid).permute(0, 2, 1, 3).reshape(n_layers, n * b, hid)
    xo = obs.permute(2, 0, 1, 3).contiguous()                                                 # (N,B,T,C)
    ref = _fp64_reference(xo, s, to_node_major(h0_ref), to_node_major(c0_ref), weights, proj)

    rows_lib = (obs * s[:, :, None, None]).permute(0, 2, 1, 3).reshape(b * n, t, c)
    layers = [tuple(weights[4 * l:4 * l + 4]) for l in range(n_layers)]
    with torch.no_grad():
        seq, (h_n, c_n) = O.lstm_library(rows_lib, layers, h0_ref, c0_ref)
    top_ref_order = ref["h_top"].reshape(n, b, hid).permute(1, 0, 2).reshape(b * n, hid)
    torch.testing.assert_close(top_ref_order, seq[:, -1], rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ref["h_n"], to_node_major(h_n), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ref["c_n"], to_node_major(c_n), rtol=1e-12, atol=1e-12)

    eps = 1e-6
    fd = torch.zeros(b, t, dtype=torch.float64)
    for bi in range(b):
        for ti in range(t):
            sp, sm = s.clone(), s.clone()
            sp[bi, ti] += eps
            sm[bi, ti] -= eps
            fd[bi, ti] = (_fp64_reference(xo, sp, to_node_major(h0_ref), to_node_major(c0_ref), weights, proj)["loss"]
                          - _fp64_reference(xo, sm, to_node_major(h0_ref), to_node_major(c0_ref), weights, proj)["loss"]) / (2 * eps)
    assert ref["d_s"].abs().max() > 1e-2
    assert_close(ref["d_s"].numpy(), fd.numpy(), "d_s vs central finite difference", 1e-7)
