"""SURVEY 8f N2: tile-major taps.  The tiled forward must be BIT-IDENTICAL to the [B,51,H,W] forward (same arithmetic,
different operand delivery), the layout conversion must be exact, and the third-generation one-channel / gray kernels
are checked against the reference-order oracle like every other forward."""
import numpy as np
import pytest
import torch

import oracle
import sstem_restoration_b200 as pkg
from tests.golden import cases

pytestmark = pytest.mark.gpu


def _cuda(*arrs):
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs)


@pytest.mark.parametrize("B,H,W", [(1, 8, 8), (2, 13, 21), (1, 64, 40)])
def test_taps_to_tiled_layout(B, H, W):
    r = np.random.default_rng(H * W)
    taps = r.standard_normal((B, 51, H, W)).astype(np.float32)
    got = pkg.taps_to_tiled(torch.from_numpy(taps).cuda()).cpu().numpy()
    ty, tx = (H + 7) // 8, (W + 7) // 8
    padded = np.zeros((B, 51, ty * 8, tx * 8), np.float32)
    padded[:, :, :H, :W] = taps
    want = padded.reshape(B, 51, ty, 8, tx, 8).transpose(0, 2, 4, 1, 3, 5)      # [b][ty][tx][tap][row][col]
    assert got.shape == (B, ty, tx, 51, 8, 8) and np.array_equal(got, want)


@pytest.mark.parametrize("B,C,H,W", [(1, 3, 64, 64), (2, 3, 37, 53), (1, 1, 40, 72), (1, 2, 16, 24), (1, 4, 24, 40), (1, 3, 7, 5)])
def test_tiled_forward_is_bit_identical_and_within_tolerance(B, C, H, W):
    inp, v, h, g = cases.sepconv_inputs(B, C, H, W, seed=300 + H + W + C, kind="unit")
    ti, tv, th = _cuda(inp, v, h)
    got = pkg.sepconv_forward_tiled(ti, pkg.taps_to_tiled(tv), pkg.taps_to_tiled(th)).cpu().numpy()
    ref32, ref64 = oracle.sepconv_forward_reforder(inp, v, h), oracle.sepconv_forward_f64(inp, v, h)
    assert np.abs(got - ref32).max() <= 1e-5 and np.abs(got - ref64).max() <= 1e-5
    nchw = pkg.SeparableConvolution.apply(ti, tv, th).cpu().numpy()
    assert np.abs(got - nchw).max() <= 2e-6                     # same math; small shapes run generation 1 on the NCHW side


def test_tiled_forward_bit_identical_at_training_size_and_gray():
    """16x3x512^2 runs the persistent kernel on both sides: identical operation order -> identical bits; gray x3 too."""
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(8)
    B, H, W = 4, 512, 512
    inp = torch.rand((B, 3, H + 50, W + 50), device=dev, generator=gen)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    vt, ht = pkg.taps_to_tiled(v), pkg.taps_to_tiled(h)
    assert torch.equal(pkg.sepconv_forward_tiled(inp, vt, ht), pkg.SeparableConvolution.apply(inp, v, h))
    gray = inp[:, :1].expand(B, 3, H + 50, W + 50).contiguous()
    general = pkg.SeparableConvolution.apply(gray, v, h)
    pkg.set_gray_replicated("assert")
    try:
        assert torch.equal(pkg.SeparableConvolution.apply(gray, v, h), general)          # generation 1, one channel
        assert torch.equal(pkg.sepconv_forward_tiled(gray, vt, ht), general)             # persistent one-channel kernel
    finally:
        pkg.set_gray_replicated("off")


def test_one_channel_persistent_kernel_vs_oracle_order():
    """C = 1 at 2x1024^2 on [B,51,H,W] taps (generation 1: the persistent one-channel kernel runs on tile-major taps only):
    exact gather with one-hot taps + linearity-free oracle check on a crop."""
    dev = "cuda"
    B, H, W = 2, 1024, 1024
    torch.manual_seed(3)
    inp = torch.rand((B, 1, H + 50, W + 50), device=dev)
    gen = torch.Generator(device="cpu").manual_seed(17)
    fy = torch.randint(0, 51, (B, 1, H, W), generator=gen).to(dev)
    fx = torch.randint(0, 51, (B, 1, H, W), generator=gen).to(dev)
    v = torch.zeros((B, 51, H, W), device=dev).scatter_(1, fy, 1.0)
    h = torch.zeros((B, 51, H, W), device=dev).scatter_(1, fx, 1.0)
    out = pkg.SeparableConvolution.apply(inp, v, h)
    yy = torch.arange(H, device=dev).view(1, 1, H, 1) + fy
    xx = torch.arange(W, device=dev).view(1, 1, 1, W) + fx
    expect = inp.reshape(B, 1, -1).gather(2, (yy * (W + 50) + xx).reshape(B, 1, -1)).reshape(B, 1, H, W)
    assert torch.equal(out, expect)
    vs = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    hs = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    got = pkg.SeparableConvolution.apply(inp, vs, hs)[0, :, 500:532, 700:764].cpu().numpy()
    ci = inp[0:1, :, 500:500 + 82, 700:700 + 114].cpu().numpy()
    ref = oracle.sepconv_forward_reforder(ci, vs[0:1, :, 500:532, 700:764].cpu().numpy().copy(), hs[0:1, :, 500:532, 700:764].cpu().numpy().copy())
    assert np.abs(got - ref[0]).max() <= 1e-5


@pytest.mark.parametrize("B,C,H,W,gray", [(1, 3, 64, 64, False), (2, 3, 37, 53, False), (1, 3, 40, 72, True), (1, 1, 24, 40, False)])
def test_tiled_interpolation_tail_matches_fused_tail_and_oracle(B, C, H, W, gray):
    """IFNet's tail (model_interp.py:90-97) on tile-major taps: frame_mean_pad + two one-plane tiled forwards, the second
    accumulating -- against the fused NCHW tail and the oracle of the unfused expression."""
    r = np.random.default_rng(B * 100 + H + W)
    i1 = r.random((B, C, H, W), dtype=np.float32)
    i2 = r.random((B, C, H, W), dtype=np.float32)
    if gray:
        i1[:, 1:] = i1[:, :1]
        i2[:, 1:] = i2[:, :1]
    taps = [cases.sepconv_inputs(B, 1, H, W, seed=40 + k, kind="unit")[1] for k in range(4)]       # k1v, k1h, k2v, k2h
    ti1, ti2 = _cuda(i1, i2)
    tt = _cuda(*taps)
    pkg.set_gray_replicated("assert" if gray else "off")
    try:
        got = pkg.interpolation_tail_tiled(ti1, ti2, *(pkg.taps_to_tiled(t) for t in tt))
        fused = pkg.interpolation_tail(ti1, ti2, *tt)
    finally:
        pkg.set_gray_replicated("off")
    want = oracle.interp_tail_reference(i1, i2, *taps)
    assert got.shape == (B, 1, H, W)
    assert np.abs(got.cpu().numpy() - want).max() <= 1e-5
    assert (got - fused).abs().max().item() <= 4e-6
    # frame_mean_pad alone: ReplicationPad2d(25) of the channel mean, views of the x6 network input accepted as they are
    x6 = torch.cat([ti1, ti2], 1) if C == 3 else None
    if x6 is not None:
        p = pkg.frame_mean_pad(x6[:, 3:6], 25, gray=False)
        ref = torch.nn.functional.pad(ti2.mean(1, keepdim=True), (25, 25, 25, 25), mode="replicate")
        assert (p - ref).abs().max().item() <= 2e-7


def test_tiled_tail_at_stack_size_and_accumulate_flag():
    """2048^2 (persistent kernel on every tile) and the accumulate flag on its own: out += forward."""
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(21)
    H = W = 1024
    i1 = torch.rand((1, 3, H, W), device=dev, generator=gen)
    i2 = torch.rand((1, 3, H, W), device=dev, generator=gen)
    taps = [torch.softmax(torch.randn((1, 51, H, W), device=dev, generator=gen), 1) for _ in range(4)]
    tiled = [pkg.taps_to_tiled(t) for t in taps]
    got = pkg.interpolation_tail_tiled(i1, i2, *tiled)
    fused = pkg.interpolation_tail(i1, i2, *taps)
    assert (got - fused).abs().max().item() <= 4e-6
    p = pkg.frame_mean_pad(i1)
    a = pkg.sepconv_forward_tiled(p, tiled[0], tiled[1])
    b = pkg.sepconv_forward_tiled(p, tiled[0], tiled[1], out=a.clone(), accumulate=True)
    assert torch.equal(b, a + a)
    with pytest.raises(ValueError):
        pkg.sepconv_forward_tiled(p, tiled[0], tiled[1], accumulate=True)
