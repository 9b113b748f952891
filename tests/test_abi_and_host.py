"""CPU tests: the C-ABI library loads and exports every symbol include/stmgcn_b200.h declares (argument counts
match the ctypes binding), and the host-side mirror of the reference modules behaves like the reference
(constructor signatures, state_dict keys/shapes, same-seed init, support construction, weight packing)."""
import os
import re

import numpy as np
import pytest
import torch
from torch import nn

from helpers import assert_close, load_golden

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_prototypes():
    text = open(os.path.join(REPO, "include", "stmgcn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(?:int32_t|int64_t|const char\*)\s+(stmgcn_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    return protos


def test_library_exports_every_declared_symbol():
    from stmgcn_b200 import _lib
    protos = _header_prototypes()
    assert len(protos) >= 20
    bound = {name: len(args) for name, _, args in _lib.SIGNATURES}
    assert set(protos) == set(bound), set(protos) ^ set(bound)
    for name, n_args in protos.items():
        assert hasattr(_lib.lib, name), f"{name} not exported by libstmgcn_b200.so"
        assert bound[name] == n_args, f"{name}: header has {n_args} args, binding has {bound[name]}"
    assert _lib.lib.stmgcn_abi_version() == _lib.ABI_VERSION
    assert _lib.lib.stmgcn_launch_count() >= 0


def test_c_abi_argument_errors_come_back_as_codes_with_a_message():
    """The C entry points validate their arguments before touching CUDA: a bad call returns a negative code and
    stmgcn_last_error() explains it (no GPU needed).  Covers the entries added in ABI 3 and 4 (the LSTM's: see
    test_lstm_entries_reject_bad_arguments_before_any_cuda_call)."""
    import ctypes
    from stmgcn_b200 import _lib
    lib = _lib.lib
    null = ctypes.c_void_p(0)
    # tensor-core projection: each entry runs its kernels or rejects the call (no quiet FFMA fallback).  The fake device
    # pointers are never dereferenced: validation fails first.
    ok, odd = ctypes.c_void_p(256), ctypes.c_void_p(4)
    err_arg, err_shape, err_align = -1, -2, -3

    def fwd_tc(ks=3, s=ok, out=ok):
        return lib.stmgcn_proj_fwd_tc(s, 128 * 64, ks, 128, ok, null, _lib.ACT_RELU, out, null)

    def bwd_tc(ks=3, s=ok, u=ok):
        return lib.stmgcn_proj_bwd_tc(s, 128 * 64, ks, 128, ok, _lib.ACT_RELU, ok, ok, ok, ok, null, u, 128 * 64, null)

    for name, call, null_arg in (("proj_fwd_tc", fwd_tc, "out"), ("proj_bwd_tc", bwd_tc, "u")):
        for kwargs, code in (({"ks": 9}, err_shape), ({null_arg: null}, err_arg), ({"s": odd}, err_align)):
            assert call(**kwargs) == code and name.encode() in lib.stmgcn_last_error(), (name, kwargs)
    # bf16 gather step: null graph; conversion: count not a multiple of 8
    rc = lib.stmgcn_cheb_spmm_step16(null, 0, 1.0, null, 0.0, null, 0.0, null, null, null, 64, null)
    assert rc < 0 and b"cheb_spmm_step16" in lib.stmgcn_last_error()
    buf = (ctypes.c_float * 16)()
    rc = lib.stmgcn_to_bf16(ctypes.addressof(buf), ctypes.addressof(buf), 12, null)
    assert rc < 0 and b"multiple of 8" in lib.stmgcn_last_error()


def test_lstm_entries_reject_bad_arguments_before_any_cuda_call():
    """One LSTM entry per kernel family and direction runs the whole recurrence (ABI 5).  Each rejects a null required
    pointer (ERR_ARG), a shape out of range (ERR_SHAPE) and, in the backward, a missing dx workspace with L > 1 (ERR_ARG),
    with a message naming the entry -- before any CUDA call (no GPU needed; the fake device pointers are never read)."""
    import ctypes
    from stmgcn_b200 import _lib
    lib = _lib.lib
    null, ok = ctypes.c_void_p(0), ctypes.c_void_p(256)
    err_arg, err_shape = -1, -2
    n_layers, t_len, rows, c_in, b_inner, hid = 3, 12, 128, 1, 8, 64

    def arr(n):
        return _lib.ptr_array([256] * n)

    def lstm16_fwd(c=c_in, xo=ok):
        return lib.stmgcn_lstm16_fwd(t_len, n_layers, rows, c, b_inner, 2, xo, ok, arr(n_layers), arr(n_layers), ok, null,
                                     null, ok, ok, ok, null, null)

    def lstm16_bwd(t=t_len, cs=ok, dx_work=ok):
        return lib.stmgcn_lstm16_bwd(t, n_layers, rows, c_in, b_inner, 2, ok, ok, arr(n_layers), arr(n_layers), ok, null,
                                     null, ok, cs, ok, ok, ok, dx_work, ok, ok, ok, ok, arr(4 * n_layers), null)

    def lstm_fwd(h=hid, hs=ok):
        return lib.stmgcn_lstm_fwd(t_len, n_layers, rows, h, c_in, b_inner, ok, ok, ok, arr(n_layers), arr(n_layers), null,
                                   null, hs, ok, null, null)

    def lstm_bwd(h=hid, gates=ok, dx_work=ok):
        return lib.stmgcn_lstm_bwd(t_len, n_layers, rows, h, c_in, b_inner, ok, ok, ok, arr(n_layers), null, null, ok, ok,
                                   gates, ok, ok, ok, dx_work, ok, ok, arr(n_layers), arr(n_layers), null)

    for name, call, cases in (
            ("lstm16_fwd", lstm16_fwd, (({"xo": null}, err_arg), ({"c": 5}, err_shape))),
            ("lstm16_bwd", lstm16_bwd, (({"cs": null}, err_arg), ({"t": 65}, err_shape), ({"dx_work": null}, err_arg))),
            ("lstm_fwd", lstm_fwd, (({"hs": null}, err_arg), ({"h": 130}, err_shape))),
            ("lstm_bwd", lstm_bwd, (({"gates": null}, err_arg), ({"h": 130}, err_shape), ({"dx_work": null}, err_arg)))):
        for kwargs, code in cases:
            assert call(**kwargs) == code and name.encode() + b":" in lib.stmgcn_last_error(), (name, kwargs)


def test_no_cpu_fallback_is_loud():
    import GCN
    from stmgcn_b200 import ops
    layer = GCN.GCN(K=2, input_dim=3, hidden_dim=4)
    with pytest.raises(RuntimeError, match="CUDA"):
        layer(torch.eye(5).repeat(2, 1, 1), torch.randn(1, 5, 3))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.obs_to_node_major(torch.randn(2, 3, 4, 1))


def test_product_code_never_imports_the_oracle():
    pat = re.compile(r"^\s*(import|from)\s+[^#\n]*oracle", re.M)
    root = os.path.join(REPO, "st-mgcn_b200", "stmgcn_b200")
    files = [os.path.join(root, fn) for fn in os.listdir(root) if fn.endswith(".py")]
    files += [os.path.join(REPO, fn) for fn in ("GCN.py", "STMGCN.py")]
    for path in files:
        assert not pat.search(open(path).read()), f"{path} imports the oracle"


@pytest.mark.parametrize("name", ["cfg1_ref", "ragged_ref", "cfg3_small_ref"])
def test_state_dict_surface_and_same_seed_init(name):
    """Same ctor keywords as Main.py:62-63; state_dict keys/shapes equal the reference's; constructing under
    the same seed reproduces the reference's parameters bit for bit (parameter creation order preserved)."""
    import STMGCN
    meta, params, _, _, _, _ = load_golden(name)
    seed = {"cfg1_ref": 0, "ragged_ref": 1, "cfg3_small_ref": 2}[name]
    torch.manual_seed(seed)
    model = STMGCN.ST_MGCN(M=meta["m"], seq_len=meta["t"], n_nodes=meta["n"], input_dim=meta["c"],
                           lstm_hidden_dim=meta["hid"], lstm_num_layers=meta["layers"], gcn_hidden_dim=meta["gcn_hid"],
                           sta_kernel_config={"kernel_type": "chebyshev", "K": meta["k"]}, gconv_use_bias=True,
                           gconv_activation=nn.ReLU)
    assert model.__class__.__name__ == "ST_MGCN"            # Model_Trainer.py:11,34 dispatches on it
    sd = model.state_dict()
    assert list(sd.keys()) == list(params.keys())
    for key in params:
        assert tuple(sd[key].shape) == tuple(params[key].shape), key
        assert torch.equal(sd[key], params[key]), f"same-seed init differs for {key}"
    model.load_state_dict(params)                            # checkpoints interchange
    assert len(model.init_hidden_list(2)) == meta["m"]
    assert STMGCN.ST_MGCN.get_support_K({"kernel_type": "chebyshev", "K": 3}) == 4
    assert STMGCN.ST_MGCN.get_support_K({"kernel_type": "localpool", "K": 1}) == 1
    with pytest.raises(ValueError):
        STMGCN.ST_MGCN.get_support_K({"kernel_type": "nope", "K": 1})


@pytest.mark.parametrize("name", ["cfg1_ref", "ragged_ref", "cfg3_small_ref"])
def test_adj_preprocessor_equals_reference_supports(name):
    import GCN
    meta, _, _, supports, adjs, _ = load_golden(name)
    pre = GCN.Adj_Preprocessor(kernel_type="chebyshev", K=meta["k"])       # Main.py:51 calls it with **config
    for a, s in zip(adjs, supports):
        got = pre.process(a)
        assert got.shape == s.shape
        assert_close(got.numpy(), s.numpy(), "dense supports", 1e-6)
        sparse = pre.process_sparse(a)
        assert len(sparse) == meta["k"] + 1 and tuple(sparse.shape) == tuple(s.shape)
        assert_close(sparse.laplacian_dense().numpy(), s[1].numpy(), "sparse L~", 1e-6)
    assert GCN.Adj_Preprocessor("localpool", 7).K == 1
    with pytest.raises(ValueError):
        GCN.Adj_Preprocessor("bogus", 2)


def test_lambda_max_options():
    import GCN
    from stmgcn_b200 import synth
    a = synth.make_adjacency(40, 0, 0.2)
    ref = GCN.Adj_Preprocessor("chebyshev", 2).process(a)
    lam = float(torch.linalg.eigvalsh((torch.eye(40) - GCN.Adj_Preprocessor.symmetric_normalize(a)).double()).max())
    pw = GCN.Adj_Preprocessor("chebyshev", 2, lambda_max="power")
    got = pw.process(a)
    want = (2.0 / lam) * (torch.eye(40) - GCN.Adj_Preprocessor.symmetric_normalize(a)) - torch.eye(40)
    assert_close(got[1].numpy(), want.numpy(), "power-iteration lambda_max", 1e-3)
    assert not torch.allclose(got[1], ref[1])
    sp_ = pw.process_sparse(a)
    assert_close(sp_.laplacian_dense().numpy(), got[1].numpy(), "sparse with lambda_max", 1e-3)


def test_lstm_weight_packing_roundtrip():
    """pack (nn.LSTM layout -> gate-interleaved K-major operands) and the gradient unpack are inverse views."""
    from stmgcn_b200 import ops
    hid, c_in, lyr = 8, 2, 3
    gen = torch.Generator().manual_seed(0)
    ws = []
    for l in range(lyr):
        in_l = c_in if l == 0 else hid
        ws += [torch.randn(4 * hid, in_l, generator=gen), torch.randn(4 * hid, hid, generator=gen),
               torch.randn(4 * hid, generator=gen), torch.randn(4 * hid, generator=gen)]
    wx, wp, bp, wpt = ops._pack_lstm(ws, lyr, hid)
    # column 4*unit+gate of the packed operand is row gate*hid+unit of the nn.LSTM matrix
    for unit in (0, 3, 7):
        for gate in range(4):
            assert torch.equal(wx[:, 4 * unit + gate], ws[0][gate * hid + unit, :])
            assert torch.equal(wp[0][:, 4 * unit + gate], ws[1][gate * hid + unit, :])
            assert torch.equal(wp[1][:hid, 4 * unit + gate], ws[4][gate * hid + unit, :])
            assert torch.equal(wp[1][hid:, 4 * unit + gate], ws[5][gate * hid + unit, :])
            assert float(bp[2][4 * unit + gate]) == pytest.approx(float(ws[10][gate * hid + unit] + ws[11][gate * hid + unit]))
    assert torch.equal(wpt[1], wp[1].t())
    grads = ops._unpack_lstm_grads(wx, wp, [b.clone() for b in bp], lyr, hid, c_in)
    assert torch.equal(grads[0], ws[0]) and torch.equal(grads[1], ws[1])
    assert torch.equal(grads[4], ws[4]) and torch.equal(grads[5], ws[5])
    assert torch.allclose(grads[2], ws[2] + ws[3])


@pytest.mark.parametrize("rows", [128, 300, 1])
def test_tile_blocked_layout_roundtrip_and_formula(rows):
    """to_blocked / from_blocked are inverse, pad to whole 128-row tiles, and place element (r, u) where the kernels'
    ws_off() expects it: (((r/128)*16 + u/4)*128 + r%128)*4 + u%4  (include/stmgcn_b200.h, stmgcn_lstm16_fwd)."""
    from stmgcn_b200 import ops
    gen = torch.Generator().manual_seed(rows)
    x = torch.randn(2, rows, 64, generator=gen)
    blk = ops.to_blocked(x)
    rp = ((rows + 127) // 128) * 128
    assert blk.shape == (2, rp, 64) and blk.is_contiguous()
    assert torch.equal(ops.from_blocked(blk, rows), x)
    flat = blk.reshape(2, -1)
    for r, u in [(0, 0), (rows - 1, 63), (rows // 2, 9), (min(rows - 1, 127), 8)]:
        off = (((r // 128) * 16 + u // 4) * 128 + r % 128) * 4 + u % 4
        assert float(flat[1, off]) == float(x[1, r, u])
    if rp != rows:                                           # padding rows are zero
        back = ops.from_blocked(blk, rp)
        assert float(back[:, rows:].abs().max()) == 0.0


def test_environment_switches_in_readme_exist_in_the_sources():
    """Every STMGCN_* switch the README advertises is read somewhere in the product code (and vice versa for the
    switches that change which kernel runs)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    readme = open(os.path.join(root, "README.md")).read()
    advertised = set(re.findall(r"`(STMGCN_[A-Z_0-9]+)=", readme))
    src = ""
    for d, _, files in os.walk(os.path.join(root, "st-mgcn_b200")):
        if os.sep + "build" in d or "__pycache__" in d:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src += open(os.path.join(d, f)).read()
    used = set(re.findall(r'"(STMGCN_[A-Z_0-9]+)"', src))
    assert advertised, "README lists no switches"
    missing = advertised - used
    assert not missing, f"README advertises switches the code never reads: {sorted(missing)}"
    kernel_switches = {s for s in used if not s.startswith(("STMGCN_DBG", "STMGCN_TC_PROFILE"))}
    undocumented = kernel_switches - advertised
    assert not undocumented, f"switches missing from README: {sorted(undocumented)}"


def test_synthetic_workloads_match_survey_table():
    from stmgcn_b200 import synth
    w = synth.WORKLOADS["cfg3"]
    assert (w.n_regions, w.n_graphs, w.cheb_order, w.seq_len, w.batch) == (4096, 3, 3, 12, 64)
    assert w.region_timesteps == 3_145_728
    a = synth.make_adjacency(64, 0, 0.10)
    assert torch.equal(a, a.t()) and float(a.diagonal().sum()) == 0 and float(a.sum(1).min()) >= 2
    x, y = synth.make_inputs(synth.WORKLOADS["cfg1"])
    assert tuple(x.shape) == (8, 4, 64, 1) and tuple(y.shape) == (8, 64, 1)
