"""CPU tests of the oracle (test infrastructure): pinned against the golden vectors generated from the
unmodified reference (tests/golden/*.npz, oracle/make_golden.py) and against closed-form known answers."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import stmgcn_oracle as O
from helpers import TOL, assert_close, load_golden


@pytest.mark.parametrize("name", ["cfg1_ref", "ragged_ref", "cfg3_small_ref"])
def test_dense_oracle_matches_reference_golden(name):
    meta, params, grads, supports, adjs, blob = load_golden(name)
    x, y = torch.from_numpy(blob["x"]), torch.from_numpy(blob["y"])
    out, loss, g = O.dense_loss_and_grads(params, x, y, supports)
    assert_close(out.numpy(), blob["out"], "forward", 1e-5)
    assert abs(float(loss) - float(blob["loss"])) < 1e-6
    for key in grads:
        assert_close(g[key].numpy(), grads[key], f"grad {key}", 2e-5)
    # support construction (GCN.py:57-97) restated
    for a, s in zip(adjs, supports):
        assert_close(O.chebyshev_supports_dense(a, meta["k"]).numpy(), s.numpy(), "supports", 1e-6)


@pytest.mark.parametrize("name", ["cfg1_ref", "ragged_ref", "cfg3_small_ref"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sparse_oracle_matches_reference_golden(name, dtype):
    """Recurrence-on-features + hand-written backward == the reference's dense forward + autograd."""
    meta, params, grads, supports, _, blob = load_golden(name)
    orc = O.SparseOracle({k: v.numpy() for k, v in params.items()},
                         [O.laplacian_csr_from_supports(s) for s in supports], meta["k"] + 1, dtype=dtype)
    out, loss, g = orc.loss_and_grads(blob["x"], blob["y"])
    assert_close(out, blob["out"], "forward", 1e-5)
    assert abs(loss - float(blob["loss"])) < 1e-5
    for key in grads:
        assert_close(g[key], grads[key], f"grad {key}", 2e-5)


def test_lstm_explicit_equals_library_lstm():
    gen = torch.Generator().manual_seed(0)
    layers = []
    for l in range(3):
        in_l = 2 if l == 0 else 8
        layers.append(tuple(torch.randn(*s, generator=gen) * 0.3 for s in ((32, in_l), (32, 8), (32,), (32,))))
    x = torch.randn(5, 7, 2, generator=gen)
    h0, c0 = torch.randn(3, 5, 8, generator=gen), torch.randn(3, 5, 8, generator=gen)
    a, (ha, ca) = O.lstm_explicit(x, layers, h0, c0)
    b, (hb, cb) = O.lstm_library(x, layers, h0, c0)
    assert_close(a.numpy(), b.detach().numpy(), "seq", 1e-5)
    assert_close(ha.numpy(), hb.detach().numpy(), "h_n", 1e-5)
    assert_close(ca.numpy(), cb.detach().numpy(), "c_n", 1e-5)


def test_known_answer_chebyshev_eigenvector():
    """T_k(L) v = cos(k arccos(lambda)) v for an eigenvector v of a symmetric L with |lambda| <= 1."""
    n, k_ord = 12, 5
    # ring graph: A_norm has eigenvalues cos(2 pi j / n); L~ = -A_norm (lambda_max = 2)
    adj = torch.zeros(n, n)
    idx = torch.arange(n)
    adj[idx, (idx + 1) % n] = 1
    adj[(idx + 1) % n, idx] = 1
    sup = O.chebyshev_supports_dense(adj.double(), k_ord)
    j = 2
    v = torch.cos(2 * np.pi * j * idx.double() / n)
    lam = -np.cos(2 * np.pi * j / n)
    for k in range(k_ord + 1):
        want = np.cos(k * np.arccos(lam)) * v
        assert torch.allclose(sup[k] @ v, want, atol=1e-12)
    # the sparse oracle's feature recurrence gives the same
    orc = O.SparseOracle({"rnn_list.0.lstm.weight_ih_l0": np.zeros((4, 1))}, [sp.csr_matrix(sup[1].numpy())], k_ord + 1)
    st = orc._cheb_stack(orc.lap[0], v.numpy().reshape(n, 1, 1))
    for k in range(k_ord + 1):
        assert np.allclose(st[k].ravel(), np.cos(k * np.arccos(lam)) * v.numpy(), atol=1e-12)


def test_known_answer_ring_graph_spectrum():
    """Ring graph: the normalised adjacency has eigenvalues cos(2 pi j / n), so the rescaled Laplacian supports[1]
    (lambda_max = 2, GCN.py:86-93) has spectrum -cos(2 pi j / n) and supports[k] has spectrum T_k of it."""
    n, k_ord = 16, 3
    adj = torch.zeros(n, n, dtype=torch.float64)
    idx = torch.arange(n)
    adj[idx, (idx + 1) % n] = 1
    adj[(idx + 1) % n, idx] = 1
    sup = O.chebyshev_supports_dense(adj, k_ord)
    lam = np.sort(-np.cos(2 * np.pi * np.arange(n) / n))
    got = np.sort(np.linalg.eigvalsh(sup[1].numpy()))
    assert np.allclose(got, lam, atol=1e-12)
    for k in range(k_ord + 1):
        want = np.sort(np.cos(k * np.arccos(np.clip(lam, -1, 1))))
        assert np.allclose(np.sort(np.linalg.eigvalsh(sup[k].numpy())), want, atol=1e-10)


def test_known_answer_order_zero_gcn_is_a_linear_layer():
    x = torch.randn(3, 9, 4)
    w, b = torch.randn(4, 5), torch.randn(5)
    out = O.dense_gcn(torch.eye(9)[None], x, w, b, relu=False)
    assert torch.allclose(out, x @ w + b, atol=1e-6)


def test_known_answer_lstm_zero_weights():
    """Zero weights: h = sigmoid(b_o) tanh(sigmoid(b_i) tanh(b_g)) after one step."""
    hid = 3
    bias = torch.tensor([0.3] * hid + [9.9] * hid + [-0.7] * hid + [1.1] * hid)
    layers = [(torch.zeros(4 * hid, 2), torch.zeros(4 * hid, hid), bias, torch.zeros(4 * hid))]
    seq, _ = O.lstm_explicit(torch.randn(4, 1, 2), layers)
    want = torch.sigmoid(torch.tensor(1.1)) * torch.tanh(torch.sigmoid(torch.tensor(0.3)) * torch.tanh(torch.tensor(-0.7)))
    assert torch.allclose(seq, want.expand_as(seq), atol=1e-7)


def test_sparse_oracle_handles_asymmetric_laplacian_and_hypothesis_shapes():
    """Dense (autograd) vs sparse (hand backward) on random asymmetric weighted graphs, odd shapes."""
    from stmgcn_b200 import synth
    for seed, (n, m, k, t, b, c, hid, lyr, g) in enumerate([(20, 2, 4, 3, 2, 2, 8, 2, 6), (33, 1, 1, 1, 1, 1, 4, 1, 4),
                                                            (17, 3, 5, 6, 3, 1, 8, 3, 8)]):
        gen = torch.Generator().manual_seed(seed)
        adjs = [synth.make_adjacency(n, i, 0.3) * (0.2 + torch.rand(n, n, generator=gen)) for i in range(m)]
        sups = [O.chebyshev_supports_dense(a, k, lambda_max=1.6) for a in adjs]
        params = O.init_params(m, t, c, hid, lyr, g, k + 1, seed=seed)
        x, y = torch.randn(b, t, n, c, generator=gen), torch.randn(b, n, c, generator=gen)
        o1, l1, g1 = O.dense_loss_and_grads(params, x, y, sups)
        orc = O.SparseOracle({k_: v.numpy() for k_, v in params.items()},
                             [O.laplacian_csr_from_supports(s) for s in sups], k + 1, dtype=np.float64)
        o2, l2, g2 = orc.loss_and_grads(x.numpy(), y.numpy())
        assert_close(o2, o1.numpy(), "forward", 2e-5)
        for key in g1:
            assert_close(g2[key], g1[key].numpy(), f"grad {key}", 5e-5)


def test_dense_matches_reference_modules():
    """The restatement against what the unmodified reference modules computed on a small case (2 graphs, K=3, H=16, L=2,
    G=8; reference supports, init, forward and autograd gradients stored by oracle/make_golden.py)."""
    _, params, grads, sups, _, blob = load_golden("dense_check_ref")
    x, y = torch.from_numpy(blob["x"]), torch.from_numpy(blob["y"])
    o2, _, g2 = O.dense_loss_and_grads(params, x, y, sups)
    assert_close(o2.numpy(), blob["out"], "forward", 1e-5)
    for key in grads:
        assert_close(g2[key].numpy(), grads[key], f"grad {key}", 2e-5)
