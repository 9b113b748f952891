"""Operand-image cache of the tensor-core paths (ops._cached_images): a cache that never hits passes every parity test, so
these count kernel launches.  A second step with unchanged parameters skips exactly the pack kernels; an in-place update
under no_grad (an optimizer step) runs them again; a projection image packed for inference only is re-packed with its
backward image when a training forward needs it."""
import pytest
import torch

from stmgcn_b200 import _lib, ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def _tc_path():
    old = ops.lstm_path()
    ops.set_lstm_path("tc")
    yield
    ops.set_lstm_path(old)


def _launches(fn) -> int:
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def _cheb_setup(ks):
    from stmgcn_b200.graph import GraphHandle, SupportSet
    n, b, p = 37, 9, 64
    gen = torch.Generator().manual_seed(ks)
    lap = (torch.rand(n, n, generator=gen) < 0.2).float() * torch.randn(n, n, generator=gen) * 0.1
    sset = SupportSet("cheb", n, ks, [GraphHandle.from_dense((lap + lap.t()).to(DEV))], torch.device(DEV))
    x = torch.randn(n, b, p, generator=gen).to(DEV).requires_grad_(True)
    w = (torch.randn(ks * p, 64, generator=gen) * 0.1).to(DEV).requires_grad_(True)
    bias = (torch.randn(64, generator=gen) * 0.1).to(DEV).requires_grad_(True)
    return sset, x, w, bias


@pytest.mark.parametrize("ks", [3, 6])
def test_projection_images_are_packed_once_per_parameter_version(ks):
    sset, x, w, bias = _cheb_setup(ks)
    step = lambda: ops.ChebGCN.apply(x, w, bias, sset, _lib.ACT_RELU).sum().backward()
    first, second = _launches(step), _launches(step)
    assert first - second == (3 if ks > 4 else 2), (first, second)     # forward image + one backward image per 4 supports
    with torch.no_grad():
        w.add_(0.01)
    assert (_launches(step), _launches(step)) == (first, second)


def test_projection_inference_image_is_repacked_for_training():
    sset, x, w, bias = _cheb_setup(3)

    def infer():
        with torch.no_grad():
            ops.ChebGCN.apply(x.detach(), w.detach(), bias.detach(), sset, _lib.ACT_RELU)

    train_fwd = lambda: ops.ChebGCN.apply(x, w, bias, sset, _lib.ACT_RELU)
    cold_infer, hit_infer = _launches(infer), _launches(infer)
    assert cold_infer - hit_infer == 1, (cold_infer, hit_infer)         # forward image only
    repack, hit_train = _launches(train_fwd), _launches(train_fwd)
    assert repack - hit_train == 2, (repack, hit_train)                 # forward + backward image
    assert _launches(infer) == hit_infer                                 # the training entry serves inference too


def test_lstm_images_are_packed_once_per_parameter_version():
    n, b, t_len, c_in, hid, layers = 37, 4, 3, 1, 64, 3
    gen = torch.Generator().manual_seed(11)
    xo = torch.randn(n, b, t_len, c_in, generator=gen).to(DEV)
    s_gate = torch.rand(b, t_len, generator=gen).to(DEV).requires_grad_(True)
    weights = [(torch.randn(*shape, generator=gen) * 0.125).to(DEV).requires_grad_(True)
               for l in range(layers)
               for shape in ((4 * hid, c_in if l == 0 else hid), (4 * hid, hid), (4 * hid,), (4 * hid,))]
    step = lambda: ops.SharedLSTM.apply(xo, s_gate, None, None, layers, hid, False, *weights)[0].sum().backward()
    first, second = _launches(step), _launches(step)
    assert first - second == layers, (first, second)                     # one pack kernel per layer
    with torch.no_grad():
        weights[5].add_(0.01)                                            # w_hh of layer 1
    assert (_launches(step), _launches(step)) == (first, second)
