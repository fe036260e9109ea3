"""Backward of the tap branch convolutions y = relu?(conv3x3(x, W) + b) (sstem_branch_conv3x3_backward,
branch_conv3x3_backward, ModuleTapBranch(trainable=True)) against the fp64 restatement in tests/_tapconv_bwd_ref.py.

Bounds, as for the tap producer (test_gpu_tapconv_backward.py), with g = grad_out * (y > 0) and y the kernel's own forward
output (so a TF32 sign flip of y near 0 is not blamed on the backward).  Operands of products are TF32 (round to nearest),
sums fp32:
  grad_x       = conv3x3(g, W'), the forward's kernel:  |err| <= 1.05 * 2^-10 * conv3x3(|g|, |W'|) + 1e-6.
  grad_weight  = sum over pixels of g x x shifted per tap.  Longest fp32 chain L = 128 * (tiles per CTA) + CTA pairs
               (the tensor-memory accumulator over a CTA's tiles, then the pair-order sum of the partials):
                   |err| <= (1.05 * 2^-10 + L * 2^-24) * sum_p |g| |x|_shifted + 1e-6.
  grad_bias    = fp32 sum of the unrounded g: chain (pixels per thread) + 5 (shuffles) + 8 (warps) + partials,
                   |err| <= L_b * 2^-24 * sum |g| + 1e-6.
Both layouts of x and of y give bit-identical gradients, so do one call for all and one call per gradient, and repeated
runs."""
import math

import numpy as np
import pytest
import torch

import sstem_restoration_b200 as pkg
from tests import _tapconv_bwd_ref as ref

pytestmark = pytest.mark.gpu


def _tf32(t):
    u = t.contiguous().view(torch.int32)
    return ((u + 0x1000) & ~0x1FFF).view(torch.float32)


def _to_chunked(x):
    B, c, h, w = x.shape
    c8 = (c + 7) // 8 * 8
    xp = torch.zeros((B, c8, h, w), dtype=torch.float32, device=x.device)
    xp[:, :c] = _tf32(x)
    return xp.view(B, c8 // 4, 4, h, w).permute(0, 1, 3, 4, 2).contiguous()


def _chains(B, cin, h, w):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ntiles = B * math.ceil(h / 16) * math.ceil(w / 8)
    pairs = min(ntiles, sms // (2 if cin > 32 else 1))
    nbx = max(64 // B, 1)
    return 128 * math.ceil(ntiles / pairs) + pairs, math.ceil(h * w / (nbx * 256)) + 5 + 8 + B * nbx


def _inputs(B, cin, cout, h, w, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((B, cin, h, w), device="cuda", generator=gen)
    wt = torch.randn((cout, cin, 3, 3), device="cuda", generator=gen) / math.sqrt(9 * cin)
    b = 0.1 * torch.randn(cout, device="cuda", generator=gen)
    gy = torch.randn((B, cout, h, w), device="cuda", generator=gen)
    return x, wt, b, gy


def _backward(gy, y, x, wt, relu=True, chunked_in=False, chunked_out=False, need=(True, True, True)):
    cout, cin = wt.shape[:2]
    return pkg.branch_conv3x3_backward(gy, y, x, pkg.pack_branch_conv_weight_adjoint(wt) if need[0] else None, cin, cout,
                                       relu=relu, chunked_in=chunked_in, chunked_out=chunked_out, need=need)


def _check(got, g, x, wt):
    B, cin, h, w = x.shape
    gx, gw, gb = (t.cpu().numpy().astype(np.float64) for t in got)
    g, x, wt = (t.cpu().numpy() for t in (g, x, wt))
    want = ref.tap_conv3x3_backward_restated(g, x, wt, upsample=False)
    bx, bw, _ = ref.tap_conv3x3_backward_restated(np.abs(g), np.abs(x), np.abs(wt), upsample=False)
    L, Lb = _chains(B, cin, h, w)
    bounds = (1.05 * 2.0 ** -10 * bx, (1.05 * 2.0 ** -10 + L * 2.0 ** -24) * bw, Lb * 2.0 ** -24 * np.abs(g).sum(axis=(0, 2, 3)))
    for name, gr, wnt, bnd in zip(("grad_x", "grad_weight", "grad_bias"), (gx, gw, gb), want, bounds):
        assert gr.shape == wnt.shape and np.isfinite(gr).all(), name
        err = np.abs(gr - wnt)
        assert (err <= bnd + 1e-6).all(), (name, float((err / (bnd + 1e-9)).max()))


SHAPES = [(1, 64, 64, 16, 8), (2, 64, 64, 13, 9), (1, 64, 51, 37, 29), (1, 64, 64, 1, 1), (1, 64, 64, 6, 5),
          (2, 17, 33, 20, 11), (1, 8, 16, 5, 7)]


@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("B,cin,cout,h,w", SHAPES)
def test_per_layer_gradients_against_the_fp64_restatement(B, cin, cout, h, w, relu):
    x, wt, b, gy = _inputs(B, cin, cout, h, w, seed=B * 1000 + cin * 7 + cout + h * 13 + w + relu)
    y = pkg.branch_conv3x3(x, pkg.pack_branch_conv_weight(wt), b, relu=relu)
    got = _backward(gy, y, x, wt, relu=relu)
    _check(got, gy * (y > 0) if relu else gy, x, wt)


@pytest.mark.parametrize("B,cin,cout,h,w", [(2, 64, 64, 13, 9), (2, 17, 33, 20, 11), (1, 8, 16, 5, 7)])
def test_layouts_single_gradients_and_repeats_are_bit_identical(B, cin, cout, h, w):
    x, wt, b, gy = _inputs(B, cin, cout, h, w, seed=B + cin + cout + h + w)
    packed = pkg.pack_branch_conv_weight(wt)
    y = pkg.branch_conv3x3(x, packed, b)
    yc = pkg.branch_conv3x3(x, packed, b, chunked_out=True)
    xc = _to_chunked(x)
    want = _backward(gy, y, x, wt)
    for xi, ci in ((x, False), (xc, True)):
        for yi, co in ((y, False), (yc, True)):
            for a, t in zip(want, _backward(gy, yi, xi, wt, chunked_in=ci, chunked_out=co)):
                assert torch.equal(a, t), (ci, co)
    for k in range(3):
        need = tuple(i == k for i in range(3))
        single = _backward(gy, y, x, wt, need=need)
        assert all((s is None) == (not n) for s, n in zip(single, need))
        assert torch.equal(single[k], want[k])
    for a, t in zip(want, _backward(gy, y, x, wt)):
        assert torch.equal(a, t)


def test_relu_mask_follows_torch_at_zero_and_nan():
    """The mask is torch's ReLU backward (threshold_backward on the output): y == 0 passes no gradient, a NaN y passes it.
    The call with the ReLU equals, bit for bit, the call without it on the gradient torch's ReLU backward returns, for both
    layouts of y."""
    x, wt, b, gy = _inputs(1, 64, 64, 19, 13, seed=5)
    y = torch.randn_like(gy)
    y[:, :, ::3] = 0.0
    y[:, :, 1::5, ::2] = float("nan")
    yr = y.clone().requires_grad_(True)
    torch.relu(yr).backward(gy)
    g = yr.grad
    assert bool((g[y == 0] == 0).all()) and torch.equal(g[y.isnan()], gy[y.isnan()])
    masked = _backward(gy, y, x, wt, relu=True)
    plain = _backward(g, None, x, wt, relu=False)
    for a, t in zip(masked, plain):
        assert torch.equal(a, t)
    for a, t in zip(masked, _backward(gy, _to_chunked(y), x, wt, chunked_out=True)):   # chunk-major y: the same mask
        assert torch.equal(a, t)


def test_many_tiles_per_cta_against_fp32_torch_autograd():
    """x [1,64,512,512]: 2 048 tiles, ~28 per CTA pair; determinism and the bounds against torch's fp32 autograd of conv2d
    (TF32 off) fed the same masked gradient."""
    x, wt, b, gy = _inputs(1, 64, 64, 512, 512, seed=17)
    x = torch.relu(x)
    y = pkg.branch_conv3x3(x, pkg.pack_branch_conv_weight(wt), b)
    got = _backward(gy, y, x, wt)
    for _ in range(2):
        for a, t in zip(got, _backward(gy, y, x, wt)):
            assert torch.equal(a, t)
    g = gy * (y > 0)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        def torch_grads(x, wt, g):
            tx, tw, tb = x.clone().requires_grad_(True), wt.clone().requires_grad_(True), torch.zeros(wt.shape[0], device="cuda", requires_grad=True)
            torch.nn.functional.conv2d(tx, tw, tb, padding=1).backward(g)
            return tx.grad, tw.grad, tb.grad
        want = torch_grads(x, wt, g)
        bx, bw, _ = torch_grads(x.abs(), wt.abs(), g.abs())
    finally:
        torch.backends.cudnn.allow_tf32 = old
    L, Lb = _chains(1, 64, 512, 512)
    bounds = (1.05 * 2.0 ** -10 * bx, (1.05 * 2.0 ** -10 + L * 2.0 ** -24) * bw, Lb * 2.0 ** -24 * g.abs().sum((0, 2, 3)))
    for name, gr, wnt, bnd in zip(("grad_x", "grad_weight", "grad_bias"), got, want, bounds):
        err = (gr - wnt).abs()
        # the fp32 reference carries its own accumulation error
        assert bool((err <= bnd * (1 + 2.0 ** -10) + 1e-4 * (name != "grad_x") + 1e-5).all()), (name, float((err / (bnd + 1e-9)).max()))
    assert abs(float((got[1] - want[1]).mean())) <= 1e-3 * float(want[1].abs().mean())


def _reference_branch():
    nn = torch.nn
    return nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 51, 3, 1, 1),
                         nn.ReLU(), nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True), nn.Conv2d(51, 51, 3, 1, 1))


@pytest.mark.parametrize("x_grad", [True, False])
def test_trainable_module_equals_the_chain_of_layer_calls(x_grad):
    torch.manual_seed(8)
    ref_seq = _reference_branch().cuda()
    m = pkg.ModuleTapBranch(tiled=False, trainable=True).cuda()
    m.load_state_dict(ref_seq.state_dict())
    x0 = torch.relu(torch.randn((2, 64, 24, 16), device="cuda"))
    x = x0.clone().requires_grad_(x_grad)
    out = m(x)
    gout = torch.randn_like(out)
    out.backward(gout)
    # the chain: three forward layers, the producer through TapConv3x3Function, then three per-layer backward calls
    convs = [getattr(m, k) for k in ("0", "2", "4")]
    a, acts = x0, [x0]
    for i, c in enumerate(convs):
        a = pkg.branch_conv3x3(a, pkg.pack_branch_conv_weight(c.weight.detach()), c.bias.detach(), chunked_in=i > 0, chunked_out=i < 2)
        acts.append(a)
    p = getattr(m, "7")
    a3 = acts[3].clone().requires_grad_(True)
    pw, pb = p.weight.detach().clone().requires_grad_(True), p.bias.detach().clone().requires_grad_(True)
    y = pkg.TapConv3x3Function.apply(a3, pw, pb, True, False)
    assert torch.equal(y, out.detach())
    y.backward(gout)
    assert torch.equal(pw.grad, p.weight.grad) and torch.equal(pb.grad, p.bias.grad)
    g = a3.grad
    for i in (2, 1, 0):
        c = convs[i]
        need_x = i > 0 or x_grad
        gx, gw, gb = _backward(g, acts[i + 1], acts[i], c.weight.detach(), chunked_in=i > 0, chunked_out=i < 2, need=(need_x, True, True))
        assert torch.equal(gw, c.weight.grad) and torch.equal(gb, c.bias.grad), i
        g = gx
    if x_grad:
        assert torch.equal(g, x.grad)
    else:
        assert x.grad is None
    assert all(t.grad is not None for t in m.parameters())


def test_four_trainable_branches_through_the_tiled_tail_and_an_optimizer_step():
    """ModuleTapBranch(trainable=True) x 4 -> ModuleInterpolationTailTiled -> L1 loss against torch's fp32 nn.Sequential x 4
    -> interpolation_tail.  A TF32 rounding can flip a ReLU mask where an activation is near 0, and the input gradient
    sums four branches with cancellation, so the comparison is norm-wise: the relative Frobenius error of the output and of
    every gradient is within 2^-7, or within twice that of torch's own TF32 autograd (cuDNN, allow_tf32) of the same
    network against the same fp32 reference.  After one optimizer step the module repacks, and its forward equals a fresh
    module loaded from the updated state_dict."""
    dev = "cuda"
    torch.manual_seed(21)
    B, h, w, C = 1, 24, 20, 3
    H, W = 2 * h, 2 * w
    refs = [_reference_branch().to(dev) for _ in range(4)]
    mods = [pkg.ModuleTapBranch(trainable=True).to(dev) for _ in range(4)]
    for m, r in zip(mods, refs):
        m.load_state_dict(r.state_dict())
    feats = torch.relu(torch.randn((B, 64, h, w), device=dev))
    i1, i2 = torch.rand((B, C, H, W), device=dev), torch.rand((B, C, H, W), device=dev)
    xs = feats.clone().requires_grad_(True)
    out = pkg.ModuleInterpolationTailTiled()(i1, i2, *(m(xs) for m in mods))
    target = out.detach() - 1.0                 # 1 below the output: the L1 gradient is the same constant on both routes
    (out - target).abs().mean().backward()
    got = [out.detach(), xs.grad] + [p.grad for m in mods for p in m.parameters()]

    def torch_route(tf32):
        old = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = tf32
        try:
            for r in refs:
                r.zero_grad(set_to_none=True)
            xr = feats.clone().requires_grad_(True)
            ref_out = pkg.interpolation_tail(i1, i2, *(r(xr) for r in refs))
            (ref_out - target).abs().mean().backward()
        finally:
            torch.backends.cudnn.allow_tf32 = old
        return [ref_out.detach(), xr.grad] + [p.grad for r in refs for p in r.parameters()]
    want, tf32 = torch_route(False), torch_route(True)
    names = ["out", "x"] + [f"{i}.{k}" for i in range(4) for k, _ in mods[i].named_parameters()]

    def rel(a, b):
        return float((a - b).norm() / b.norm().clamp_min(1e-30))
    for name, a, t, ref_tf32 in zip(names, got, want, tf32):
        assert a is not None, name
        assert rel(a, t) <= max(2.0 ** -7, 2 * rel(ref_tf32, t)), (name, rel(a, t), rel(ref_tf32, t))
    opt = torch.optim.SGD([p for m in mods for p in m.parameters()], lr=0.5)
    with torch.no_grad():
        before = mods[0](feats)
    opt.step()
    with torch.no_grad():
        after = mods[0](feats)
        fresh = pkg.ModuleTapBranch().to(dev)
        fresh.load_state_dict(mods[0].state_dict())
        assert not torch.equal(before, after)
        assert torch.equal(after, fresh(feats))
