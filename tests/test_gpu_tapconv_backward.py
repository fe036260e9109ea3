"""Backward of the tap producer y = conv3x3(up(x), W) + b (sstem_tap_conv3x3_backward, TapConv3x3Function,
ModuleTapProducer(trainable=True)) against the fp64 restatement in tests/_tapconv_bwd_ref.py.

Bounds.  Both operands of every product are rounded to TF32 (round to nearest, relative error <= 2^-11 each), products
are accumulated in fp32, as in the forward (tests/test_gpu_tapconv.py):
  grad_x       = up^T(conv3x3(gy, W')).  The convolution is the forward's kernel, so its error is at most
               1.05 * 2^-10 * conv3x3(|gy|, |W'|); up^T has non-negative weights and adds fp32 roundings only, so
                   |err| <= 1.05 * 2^-10 * up^T(conv3x3(|gy|, |W'|)) + 1e-6.
  grad_weight  = sum over pixels of gy * U, U = up(x) blended in fp32 and rounded to TF32 (|U| <= up(|x|)).  The longest
               fp32 accumulation chain is L = 128 * (tiles per CTA) + CTAs (a CTA's tensor-memory accumulator over its
               tiles, then the CTA-order sum of the partials), so
                   |err| <= (1.05 * 2^-10 + L * 2^-24) * sum_p |gy| * up(|x|)_shifted + 1e-6.
  grad_bias    = fp32 sum of gy: chain (tiles per CTA) + 128 + CTAs, |err| <= L_b * 2^-24 * sum |gy| + 1e-6.
NCHW and tile-major gy give bit-identical gradients; repeated runs are bit-identical."""
import math
import os

import numpy as np
import pytest
import torch

import sstem_restoration_b200 as pkg
from tests import _tapconv_bwd_ref as ref

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _chains(B, H, W):
    ntiles = B * math.ceil(H / 16) * math.ceil(W / 8)
    ctas = min(ntiles, torch.cuda.get_device_properties(0).multi_processor_count)
    per = math.ceil(ntiles / ctas)
    return 128 * per + ctas, per + 128 + ctas


def _grads(x, w, b, gy, ups, tiled=False):
    """(grad_x, grad_weight, grad_bias) through TapConv3x3Function; gy NCHW (made tile-major here when tiled)"""
    tx = x.clone().requires_grad_(True)
    tw = w.clone().requires_grad_(True)
    tb = b.clone().requires_grad_(True)
    y = pkg.TapConv3x3Function.apply(tx, tw, tb, ups, tiled)
    y.backward(pkg.taps_to_tiled(gy) if tiled else gy)
    return tx.grad, tw.grad, tb.grad


def _check(got, x, w, gy, ups):
    gx, gw, gb = (t.cpu().numpy().astype(np.float64) for t in got)
    x, w, gy = (t.cpu().numpy() for t in (x, w, gy))
    want = ref.tap_conv3x3_backward_restated(gy, x, w, ups)
    bx, bw, _ = ref.tap_conv3x3_backward_restated(np.abs(gy), np.abs(x), np.abs(w), ups)
    L, Lb = _chains(gy.shape[0], gy.shape[2], gy.shape[3])
    bounds = (1.05 * 2.0 ** -10 * bx, (1.05 * 2.0 ** -10 + L * 2.0 ** -24) * bw,
              Lb * 2.0 ** -24 * np.abs(gy).sum(axis=(0, 2, 3)))
    for name, g, wnt, bnd in zip(("grad_x", "grad_weight", "grad_bias"), (gx, gw, gb), want, bounds):
        assert g.shape == wnt.shape and np.isfinite(g).all(), name
        err = np.abs(g - wnt)
        assert (err <= bnd + 1e-6).all(), (name, float((err / (bnd + 1e-9)).max()))


def _inputs(B, cin, cout, h, w, ups, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    H, W = (2 * h, 2 * w) if ups else (h, w)
    x = torch.relu(torch.randn((B, cin, h, w), device="cuda", generator=gen))
    wt = torch.randn((cout, cin, 3, 3), device="cuda", generator=gen) / math.sqrt(9 * cin)
    b = 0.1 * torch.randn(cout, device="cuda", generator=gen)
    gy = torch.randn((B, cout, H, W), device="cuda", generator=gen)
    return x, wt, b, gy


@pytest.mark.parametrize("B,cin,cout,h,w,ups", [
    (1, 51, 51, 8, 4, True), (2, 51, 51, 13, 9, True), (1, 51, 51, 1, 1, True), (1, 51, 51, 1, 7, True),
    (2, 51, 51, 6, 1, True), (2, 8, 16, 5, 3, True), (1, 52, 52, 6, 5, True), (1, 3, 5, 9, 6, False),
    (2, 17, 33, 20, 11, False), (1, 51, 51, 37, 29, False), (1, 51, 51, 1, 1, False),
])
def test_small_ragged_and_degenerate_shapes(B, cin, cout, h, w, ups):
    x, wt, b, gy = _inputs(B, cin, cout, h, w, ups, seed=B * 1000 + cin * 7 + cout + h * 13 + w)
    got = _grads(x, wt, b, gy, ups)
    _check(got, x, wt, gy, ups)
    if cout == 51:                                          # tile-major gy: the same gradients, bit for bit
        for a, t in zip(got, _grads(x, wt, b, gy, ups, tiled=True)):
            assert torch.equal(a, t)


def test_nan_in_tiled_padding_changes_nothing():
    x, wt, b, gy = _inputs(2, 51, 51, 13, 9, True, seed=4)       # 26 x 18 output: ragged 8 x 8 blocks
    want = _grads(x, wt, b, gy, True, tiled=True)
    tg = pkg.taps_to_tiled(gy)
    pad = pkg.taps_to_tiled(torch.ones_like(gy)) == 0          # entries outside the image
    assert bool(pad.any())
    tg[pad] = float("nan")
    tx, tw, tb = x.clone().requires_grad_(True), wt.clone().requires_grad_(True), b.clone().requires_grad_(True)
    pkg.TapConv3x3Function.apply(tx, tw, tb, True, True).backward(tg)
    for a, g in zip(want, (tx.grad, tw.grad, tb.grad)):
        assert torch.equal(a, g)


def test_determinism_with_many_tiles_per_cta():
    """2 x 256 x 256 output = 1024 tiles over the SMs: several tiles per CTA, partials of every CTA in the sum."""
    x, wt, b, gy = _inputs(2, 51, 51, 128, 128, True, seed=9)
    a = _grads(x, wt, b, gy, True)
    _check(a, x, wt, gy, True)
    for _ in range(2):
        for u, v in zip(a, _grads(x, wt, b, gy, True)):
            assert torch.equal(u, v)


def test_large_image_against_fp32_torch_autograd():
    """1024^2 output (8192 tiles): torch's own fp32 autograd (TF32 off) of interpolate + conv2d on the same GPU, the same
    bounds computed with torch from absolute values, and no systematic offset."""
    x, wt, b, gy = _inputs(1, 51, 51, 512, 512, True, seed=77)
    got = _grads(x, wt, b, gy, True)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        def torch_grads(x, wt, b, gy):
            tx, tw, tb = (t.clone().requires_grad_(True) for t in (x, wt, b))
            up = torch.nn.functional.interpolate(tx, scale_factor=2, mode="bilinear", align_corners=True)
            torch.nn.functional.conv2d(up, tw, tb, padding=1).backward(gy)
            return tx.grad, tw.grad, tb.grad
        want = torch_grads(x, wt, b, gy)
        bx, bw, _ = torch_grads(x.abs(), wt.abs(), b, gy.abs())
    finally:
        torch.backends.cudnn.allow_tf32 = old
    L, Lb = _chains(1, 1024, 1024)
    bounds = (1.05 * 2.0 ** -10 * bx, (1.05 * 2.0 ** -10 + L * 2.0 ** -24) * bw, Lb * 2.0 ** -24 * gy.abs().sum((0, 2, 3)))
    for name, g, wnt, bnd in zip(("grad_x", "grad_weight", "grad_bias"), got, want, bounds):
        err = (g - wnt).abs()
        # the fp32 reference carries its own accumulation error: 1e-5 absolute plus 2^-20 of the bound
        assert bool((err <= bnd * (1 + 2.0 ** -10) + 1e-4 * (name != "grad_x") + 1e-5).all()), (name, float((err / (bnd + 1e-9)).max()))
    errx = (got[0] - want[0]).abs()
    assert float(errx.mean()) <= 0.1 * float((2.0 ** -10 * bx).mean())
    assert abs(float((got[0] - want[0]).mean())) <= 1e-6
    assert abs(float((got[1] - want[1]).mean())) <= 1e-3 * float(want[1].abs().mean())


def test_reference_model_layer_golden():
    g = np.load(os.path.join(GOLDEN, "tap_producer_ref.npz"))
    x, wt, b = (torch.from_numpy(g[k]).cuda() for k in ("x", "weight", "bias"))
    gy = torch.randn(tuple(g["y"].shape), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2024))
    _check(_grads(x, wt, b, gy, True), x, wt, gy, True)


def test_trainable_producers_through_the_tiled_tail():
    """ModuleTapProducer(tiled=True, trainable=True) x 4 -> ModuleInterpolationTailTiled -> L1 loss, against
    interpolate + conv2d (torch fp32) -> interpolation_tail.  The target sits 1 below the output, so the L1 gradient is
    the same constant on both routes; the tap gradients the tail returns then differ only through the forward taps
    (TF32 here), by at most another 1.05 * 2^-10 of the same magnitudes: the bound is twice the layer's."""
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(31)
    B, h, w, C = 1, 40, 36, 3
    H, W = 2 * h, 2 * w
    acts = [torch.relu(torch.randn((B, 51, h, w), device=dev, generator=gen)) for _ in range(4)]
    i1 = torch.rand((B, C, H, W), device=dev, generator=gen)
    i2 = torch.rand((B, C, H, W), device=dev, generator=gen)
    mods = [pkg.ModuleTapProducer(tiled=True, trainable=True).to(dev) for _ in range(4)]
    with torch.no_grad():
        for m in mods:
            m.weight.div_(4.0)
            m.bias.normal_(0.0, 0.02, generator=gen)
    xs = [a.clone().requires_grad_(True) for a in acts]
    out = pkg.ModuleInterpolationTailTiled()(i1, i2, *(m(x) for m, x in zip(mods, xs)))
    target = out.detach() - 1.0
    (out - target).abs().mean().backward()

    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        convs, xr = [], [a.clone().requires_grad_(True) for a in acts]
        for m in mods:
            c = torch.nn.Conv2d(51, 51, 3, 1, 1).to(dev)
            c.load_state_dict({"weight": m.weight.detach(), "bias": m.bias.detach()})
            convs.append(c)
        taps = [c(torch.nn.functional.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)) for c, x in zip(convs, xr)]
        ref_out = pkg.interpolation_tail(i1, i2, *taps)
        for t in taps:
            t.retain_grad()
        (ref_out - target).abs().mean().backward()
        bounds = []
        for c, x, t in zip(convs, acts, taps):
            tx, tw = x.clone().requires_grad_(True), c.weight.detach().abs().requires_grad_(True)
            up = torch.nn.functional.interpolate(tx, scale_factor=2, mode="bilinear", align_corners=True)
            torch.nn.functional.conv2d(up, tw, padding=1).backward(t.grad.abs())
            bounds.append((tx.grad.abs(), tw.grad, t.grad.abs().sum((0, 2, 3))))
    finally:
        torch.backends.cudnn.allow_tf32 = old
    L, Lb = _chains(B, H, W)
    for m, x, c, xrr, (bx, bw, bb) in zip(mods, xs, convs, xr, bounds):
        for g, wnt, bnd in ((x.grad, xrr.grad, 2 * 1.05 * 2.0 ** -10 * bx), (m.weight.grad, c.weight.grad, (2 * 1.05 * 2.0 ** -10 + L * 2.0 ** -24) * bw),
                            (m.bias.grad, c.bias.grad, (2.0 ** -10 + Lb * 2.0 ** -24) * bb)):
            err = (g - wnt).abs()
            assert bool((err <= bnd + 1e-7).all()), float((err / (bnd + 1e-12)).max())
