"""Tap branch convolutions (branch_conv3x3, ModuleTapBranch): Conv2d(cin <= 64, cout <= 64, 3, 1, 1) -> ReLU on tcgen05.

Parity bar, per layer, as for the tap producer (test_gpu_tapconv.py): operands rounded to TF32, fp32 accumulation, so

    |got - relu(fp64 oracle)| <= 1.05 * 2^-10 * (conv(|x|, |w|) + |bias|) + 1e-6

on every element (ReLU is 1-Lipschitz, so the bound survives it).  Between the input layouts, the output layouts and from
run to run the results must be bit-identical."""
import numpy as np
import pytest
import torch

import oracle
import sstem_restoration_b200 as pkg

pytestmark = pytest.mark.gpu


def _tf32(t):
    """cvt.rna.tf32.f32 on the host side: round the magnitude to 10 mantissa bits, ties away from zero."""
    u = t.contiguous().view(torch.int32)
    return ((u + 0x1000) & ~0x1FFF).view(torch.float32)


def _to_chunked(x):
    """[B, c, h, w] -> chunk-major [B, C8/4, h, w, 4], TF32-rounded, padding channels 0 (what the launcher builds)."""
    B, c, h, w = x.shape
    c8 = (c + 7) // 8 * 8
    xp = torch.zeros((B, c8, h, w), dtype=torch.float32, device=x.device)
    xp[:, :c] = _tf32(x)
    return xp.view(B, c8 // 4, 4, h, w).permute(0, 1, 3, 4, 2).contiguous()


def _from_chunked(y, c):
    B, k, h, w, _ = y.shape
    return y.permute(0, 1, 4, 2, 3).reshape(B, 4 * k, h, w)[:, :c]


def _check(got, x, w, b, relu):
    want = oracle.tap_conv3x3_restated(x, w, b, upsample=False)
    if relu:
        want = np.maximum(want, 0)
    bound = oracle.tap_conv3x3_restated(np.abs(x), np.abs(w), None if b is None else np.abs(b), upsample=False)
    err = np.abs(got.astype(np.float64) - want)
    assert got.shape == want.shape
    assert np.isfinite(got).all()
    assert (err <= 1.05 * 2.0 ** -10 * bound + 1e-6).all(), float((err / (2.0 ** -10 * bound + 1e-9)).max())


SHAPES = [(1, 64, 64, 16, 8), (2, 64, 64, 13, 9), (1, 64, 51, 37, 29), (1, 64, 64, 1, 1), (1, 64, 64, 6, 5),
          (2, 17, 33, 20, 11), (1, 8, 16, 5, 7)]


@pytest.mark.parametrize("B,cin,cout,h,w", SHAPES)
def test_per_layer_bound_and_layouts(B, cin, cout, h, w):
    r = np.random.default_rng(B * 1000 + cin * 7 + cout + h * 13 + w)
    x = r.standard_normal((B, cin, h, w)).astype(np.float32)
    wt = (r.standard_normal((cout, cin, 3, 3)) / np.sqrt(9 * cin)).astype(np.float32)
    bs = r.standard_normal(cout).astype(np.float32)
    tx, packed = torch.from_numpy(x).cuda(), pkg.pack_branch_conv_weight(torch.from_numpy(wt).cuda())
    xc = _to_chunked(tx)
    for bias in (bs, None):
        tb = None if bias is None else torch.from_numpy(bias).cuda()
        for relu in (True, False):
            y = pkg.branch_conv3x3(tx, packed, tb, relu=relu)
            _check(y.cpu().numpy(), x, wt, bias, relu)
            # chunk-major input: bit-identical; two runs: bit-identical
            assert torch.equal(pkg.branch_conv3x3(xc, packed, tb, relu=relu, chunked_in=True), y)
            assert torch.equal(pkg.branch_conv3x3(tx, packed, tb, relu=relu), y)
            # chunk-major output = the NCHW output rounded to TF32, padding channels 0
            yc = pkg.branch_conv3x3(tx, packed, tb, relu=relu, chunked_out=True)
            assert yc.shape == (B, (cout + 7) // 8 * 2, h, w, 4)
            assert torch.equal(yc, _to_chunked(y))
            assert torch.equal(_from_chunked(yc, cout), _tf32(y))
            assert torch.equal(pkg.branch_conv3x3(xc, packed, tb, relu=relu, chunked_in=True, chunked_out=True), yc)


def test_many_tiles_per_cta_against_fp32_library_convolution():
    """x [1,64,512,512]: 2 048 tiles per layer, ~14 per CTA, so every barrier runs through its phases many times; the fp64
    oracle is too slow here, so the comparison is against torch's fp32 conv2d (TF32 off) on the GPU, same bound."""
    gen = torch.Generator(device="cuda").manual_seed(31)
    x = torch.relu(torch.randn((1, 64, 512, 512), device="cuda", generator=gen))
    w = torch.randn((64, 64, 3, 3), device="cuda", generator=gen) / 24.0
    b = 0.1 * torch.randn(64, device="cuda", generator=gen)
    got = pkg.branch_conv3x3(x, pkg.pack_branch_conv_weight(w), b)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        want = torch.relu(torch.nn.functional.conv2d(x, w, b, padding=1))
        bound = torch.nn.functional.conv2d(x.abs(), w.abs(), b.abs(), padding=1)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    err = (got - want).abs()
    assert bool((err <= 1.05 * 2.0 ** -10 * bound + 1e-5).all()), float((err / (2.0 ** -10 * bound + 1e-9)).max())
    assert float(err.mean()) <= 0.1 * float((2.0 ** -10 * bound).mean())


def _reference_branch():
    nn = torch.nn
    return nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 51, 3, 1, 1),
                         nn.ReLU(), nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True), nn.Conv2d(51, 51, 3, 1, 1))


def test_module_equals_the_chain_of_layer_calls_and_the_reference():
    torch.manual_seed(4)
    ref = _reference_branch().cuda()
    m = pkg.ModuleTapBranch().cuda()
    m.load_state_dict(ref.state_dict())
    mn = pkg.ModuleTapBranch(tiled=False).cuda()
    mn.load_state_dict(ref.state_dict())
    x = torch.relu(torch.randn((2, 64, 40, 24), device="cuda"))
    with torch.no_grad():
        got_tiled, got = m(x), mn(x)
    # the chain of per-layer NCHW calls, then the producer
    a = x
    for i, relu in ((0, True), (2, True), (4, True)):
        a = pkg.branch_conv3x3(a, pkg.pack_branch_conv_weight(ref[i].weight.detach()), ref[i].bias.detach(), relu=relu)
    chain = pkg.tap_conv3x3(a, pkg.pack_tap_conv_weight(ref[7].weight.detach()), ref[7].bias.detach())
    assert torch.equal(got, chain)
    assert torch.equal(got_tiled, pkg.taps_to_tiled(got))
    # the fp32 Sequential: a sanity bound on four TF32 layers
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            want = ref(x)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert float((got - want).abs().max()) <= 2.0 ** -8 * float(want.abs().max())


def test_module_repacks_after_weight_update_and_is_forward_only():
    m = pkg.ModuleTapBranch(tiled=False).cuda()
    x = torch.rand((1, 64, 16, 16), device="cuda")
    y0 = m(x)
    with torch.no_grad():
        getattr(m, "2").weight.mul_(2.0)
    y1 = m(x)
    assert not torch.equal(y0, y1)
    fresh = pkg.ModuleTapBranch(tiled=False).cuda()
    fresh.load_state_dict(m.state_dict())
    assert torch.equal(fresh(x), y1)
    with pytest.raises(NotImplementedError):
        m(x.clone().requires_grad_(True))
    with pytest.raises(NotImplementedError):
        pkg.branch_conv3x3(x.clone().requires_grad_(True), pkg.pack_branch_conv_weight(torch.rand((64, 64, 3, 3), device="cuda")))
    with torch.no_grad():
        assert m(x.clone().requires_grad_(True)).shape == (1, 51, 32, 32)
