"""CPU: the fp64 restatement of the tap producer's backward (tests/_tapconv_bwd_ref.py) is the adjoint of
oracle.tap_conv3x3_restated and agrees with torch's CPU autograd; the backward's C-ABI argument checks."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from tests import _tapconv_bwd_ref as ref

SHAPES = [(1, 3, 4, 5, 7, True), (2, 5, 3, 1, 1, True), (1, 4, 6, 1, 9, True), (2, 3, 2, 7, 1, True),
          (1, 51, 51, 4, 3, True), (2, 4, 5, 6, 5, False), (1, 3, 2, 1, 1, False)]


def _inputs(B, cin, cout, h, w, ups, seed):
    r = np.random.default_rng(seed)
    H, W = (2 * h, 2 * w) if ups else (h, w)
    return (r.standard_normal((B, cin, h, w)), r.standard_normal((cout, cin, 3, 3)), r.standard_normal(cout),
            r.standard_normal((B, cout, H, W)))


@pytest.mark.parametrize("B,cin,cout,h,w,ups", SHAPES)
def test_restated_backward_is_the_adjoint(B, cin, cout, h, w, ups):
    x, wt, b, gy = _inputs(B, cin, cout, h, w, ups, B + cin + 7 * h + w)
    gx, gw, gb = ref.tap_conv3x3_backward_restated(gy, x, wt, ups)
    y = oracle.tap_conv3x3_restated(x, wt, None, ups)
    lhs = float((y * gy).sum())
    scale = float(np.abs(oracle.tap_conv3x3_restated(np.abs(x), np.abs(wt), None, ups) * np.abs(gy)).sum())
    assert abs(lhs - float((x * gx).sum())) <= 1e-12 * scale            # <conv(up(x)), gy> = <x, grad_x>
    assert abs(lhs - float((wt * gw).sum())) <= 1e-12 * scale           # y is linear in W: <y(W), gy> = <W, grad_W>
    yb = oracle.tap_conv3x3_restated(np.zeros_like(x), wt, b, ups)
    assert abs(float((yb * gy).sum()) - float((b * gb).sum())) <= 1e-12 * float(np.abs(gy).sum() * np.abs(b).max())
    if ups:                                                             # the matrix form of up is the oracle's upsample
        assert np.abs(ref.upsample2x(x) - oracle.upsample2x_align_corners_restated(x)).max() <= 1e-12 * np.abs(x).max()


@pytest.mark.parametrize("B,cin,cout,h,w,ups", SHAPES)
def test_restated_backward_matches_torch_cpu_autograd(B, cin, cout, h, w, ups):
    x, wt, b, gy = (a.astype(np.float32) for a in _inputs(B, cin, cout, h, w, ups, 3 * B + cin + h))
    tx = torch.from_numpy(x).requires_grad_(True)
    conv = torch.nn.Conv2d(cin, cout, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(wt))
        conv.bias.copy_(torch.from_numpy(b))
    up = torch.nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)(tx) if ups else tx
    conv(up).backward(torch.from_numpy(gy))
    gx, gw, gb = ref.tap_conv3x3_backward_restated(gy, x, wt, ups)
    for got, want in ((tx.grad, gx), (conv.weight.grad, gw), (conv.bias.grad, gb)):
        got = got.numpy().astype(np.float64)
        assert got.shape == want.shape
        assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max())


def test_backward_argument_errors_do_not_need_a_gpu(built_lib):
    from sstem_restoration_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1024)
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16       # 16-byte aligned host memory
    bw = lib.sstem_tap_conv3x3_backward
    assert lib.sstem_tap_conv3x3_pack_weights_adjoint(None, p, 51, 51, None) == -1
    assert lib.sstem_tap_conv3x3_pack_weights_adjoint(p, p, 51, 53, None) == -2                  # cout <= 52
    assert lib.sstem_tap_conv3x3_pack_weights_adjoint(p, p, 53, 51, None) == -2                  # cin <= 52
    assert lib.sstem_tap_conv3x3_pack_weights_adjoint(p, p + 4, 51, 51, None) == -3              # packed 16-byte aligned
    assert lib.sstem_tap_conv3x3_pack_weights_adjoint(p, p, 51, 51, None) == -4                  # host memory
    assert bw(None, p, p, p, p, p, 1, 51, 51, 4, 4, 1, None) == -1
    assert bw(p, None, p, p, p, p, 1, 51, 51, 4, 4, 1, None) == -1
    assert bw(p, p, None, p, None, None, 1, 51, 51, 4, 4, 1, None) == -1                         # grad_x needs the adjoint image
    assert bw(p, p, p, p, p, p, 1, 51, 51, 4, 4, 4, None) == -5
    assert bw(p, p, p, p, p, p, 0, 51, 51, 4, 4, 1, None) == -2
    assert bw(p, p, p, p, p, p, 1, 51, 51, 0, 4, 1, None) == -2
    assert bw(p, p, p, p, p, p, 1, 53, 51, 4, 4, 1, None) == -2                                  # cin <= 52
    assert bw(p, p, p, p, p, p, 1, 51, 53, 4, 4, 1, None) == -2                                  # cout <= 52
    assert bw(p, p, p, p, p, p, 1, 51, 32, 4, 4, 3, None) == -2                                  # tiled: 51 taps only
    assert bw(p, p, p + 4, p, p, p, 1, 51, 51, 4, 4, 1, None) == -3
    assert bw(p + 2, p, p, p, p, p, 1, 51, 51, 4, 4, 1, None) == -3
    assert bw(p, p, p, p, p, p + 1, 1, 51, 51, 4, 4, 1, None) == -3
    assert bw(p, p, p, p, p, p, 1, 51, 51, 4, 4, 1, None) == -4                                  # host memory
    assert bw(p, p, None, None, p, None, 1, 51, 51, 4, 4, 3, None) == -4


def test_trainable_producer_refuses_cpu_tensors():
    import sstem_restoration_b200 as pkg
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(NotImplementedError):
        pkg.pack_tap_conv_weight_adjoint(torch.zeros((51, 51, 3, 3)))
    with pytest.raises(NotImplementedError):
        pkg.ModuleTapProducer(trainable=True)(torch.zeros((1, 51, 4, 4), requires_grad=True))
