"""Tap gradients on tile-major taps (sstem_sepconv_backward_tiled, SeparableConvolutionTiled, ModuleInterpolationTailTiled).

The tiled backward always runs the persistent (third-generation) tap-gradient kernel.  Where the [B,51,H,W] path runs the
same kernel, the arithmetic is the same and the gradients must be BIT-IDENTICAL; elsewhere (small shapes run generation 1
on the [B,51,H,W] side) both are held to the oracle under the sepconv protocol:
  P1  unit-scale inputs: max-abs <= 1e-5 vs the reference-order oracle;
  P2  raw N(0,1) taps: max-abs <= 1e-5 * max(1, max|ref|) AND the error vs fp64 does not exceed the reference order's own
      error (x 1.25, or 2e-6 * scale).
Every entry of a tiled gradient outside the image must be exactly 0."""
import numpy as np
import pytest
import torch

import oracle
import sstem_restoration_b200 as pkg
from sstem_restoration_b200 import _lib
from tests.golden import cases

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _cuda(*arrs):
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs)


def _check_p(got, ref32, ref64, what):
    scale = max(1.0, float(np.abs(ref64).max()))
    err_vs_ref = float(np.abs(got.astype(np.float64) - ref32).max())
    err_new = float(np.abs(got - ref64).max())
    err_ref = float(np.abs(ref32 - ref64).max())
    assert err_vs_ref <= TOL * scale, f"{what}: |new-ref|={err_vs_ref:.3e} scale={scale:.3g}"
    assert err_new <= max(err_ref * 1.25, 2e-6 * scale), f"{what}: err(new,f64)={err_new:.3e} > err(ref,f64)={err_ref:.3e}"


def _padding_mask(B, H, W, dev="cuda"):
    """True at the entries of a tile-major tensor that lie outside the image."""
    return pkg.taps_to_tiled(torch.ones((B, 51, H, W), device=dev)) == 0


def _tiled_grads(inp, v, h, g, gray=False, want=(True, True, True)):
    """-> (grad_input, grad_vertical_tiled, grad_horizontal_tiled) through the C ABI (None where not wanted)."""
    B, C, IH, IW = inp.shape
    H, W = IH - 50, IW - 50
    vt, ht = pkg.taps_to_tiled(v), pkg.taps_to_tiled(h)
    gi = torch.full_like(inp, float("nan")) if want[0] else None
    gv = torch.full_like(vt, float("nan")) if want[1] else None       # NaN: an entry the kernel does not write shows up
    gh = torch.full_like(ht, float("nan")) if want[2] else None
    code = _lib.load().sstem_sepconv_backward_tiled(
        g.data_ptr(), inp.data_ptr(), vt.data_ptr(), ht.data_ptr(), *(t.data_ptr() if t is not None else None for t in (gi, gv, gh)),
        B, C, H, W, 51, _lib.SEPCONV_GRAY_REPLICATED if gray else 0, torch.cuda.current_stream().cuda_stream)
    _lib.check(code, "sstem_sepconv_backward_tiled")
    return gi, gv, gh


def _nchw_grads(inp, v, h, g, need_input=False):
    inp = inp.clone().requires_grad_(need_input)
    v = v.clone().requires_grad_(True)
    h = h.clone().requires_grad_(True)
    pkg.SeparableConvolution.apply(inp, v, h).backward(g)
    return inp.grad, v.grad, h.grad


@pytest.mark.parametrize("B,H,W", [(1, 8, 8), (2, 13, 21), (1, 9, 40), (3, 1, 1)])
def test_taps_from_tiled_inverts_taps_to_tiled(B, H, W):
    r = np.random.default_rng(H * W + B)
    (taps,) = _cuda(r.standard_normal((B, 51, H, W)).astype(np.float32))
    tiled = pkg.taps_to_tiled(taps)
    assert torch.equal(pkg.taps_from_tiled(tiled, H, W), taps)
    garbage = tiled.clone()
    garbage[_padding_mask(B, H, W)] = float("nan")              # padding entries are not read
    assert torch.equal(pkg.taps_from_tiled(garbage, H, W), taps)


@pytest.mark.parametrize("B,C,H,W", [(4, 3, 512, 512), (1, 3, 1001, 1004), (2, 6, 512, 512)])
def test_bit_identical_to_the_nchw_persistent_kernel(B, C, H, W):
    """Shapes on which the [B,51,H,W] path runs the persistent kernel too (W % 4 == 0, enough tiles): same arithmetic,
    same bits.  1001 rows: H % 8 == 1, the last tile row is one image row and seven padding rows."""
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(B * C + H)
    inp = torch.rand((B, C, H + 50, W + 50), device=dev, generator=gen)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    g = torch.randn((B, C, H, W), device=dev, generator=gen)
    _, gv_t, gh_t = _tiled_grads(inp, v, h, g, want=(False, True, True))
    _, gv, gh = _nchw_grads(inp, v, h, g)
    assert torch.equal(pkg.taps_from_tiled(gv_t, H, W), gv)
    assert torch.equal(pkg.taps_from_tiled(gh_t, H, W), gh)
    pad = _padding_mask(B, H, W)
    assert bool((gv_t[pad] == 0).all()) and bool((gh_t[pad] == 0).all())


@pytest.mark.parametrize("kind", ["unit", "randn"])
@pytest.mark.parametrize("B,C,H,W", [(1, 1, 20, 24), (2, 2, 12, 16), (1, 3, 9, 13), (1, 4, 20, 30), (2, 3, 12, 37),
                                     (1, 3, 7, 5), (1, 5, 17, 11)])
def test_oracle_parity_at_edge_shapes(B, C, H, W, kind):
    """C = 1..5 (3-channel chunks and single planes, later ones accumulating), W % 4 != 0 (the gradient is staged),
    H % 8 in 1..4 (half a tile row of padding rows), a shape smaller than one tile."""
    inp, v, h, g = cases.sepconv_inputs(B, C, H, W, seed=700 + 10 * C + H + W, kind=kind)
    _, gv_t, gh_t = _tiled_grads(*_cuda(inp, v, h, g), want=(False, True, True))
    gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
    what = f"{kind} {B, C, H, W}"
    _check_p(pkg.taps_from_tiled(gv_t, H, W).cpu().numpy(), oracle.sepconv_grad_vertical_reforder(g, inp, h), gv64, "gv " + what)
    _check_p(pkg.taps_from_tiled(gh_t, H, W).cpu().numpy(), oracle.sepconv_grad_horizontal_reforder(g, inp, v), gh64, "gh " + what)
    pad = _padding_mask(B, H, W)
    assert bool((gv_t[pad] == 0).all()) and bool((gh_t[pad] == 0).all())


@pytest.mark.parametrize("B,C,H,W", [(2, 3, 96, 100), (1, 4, 41, 64)])
def test_single_gradient_calls_and_grad_input(B, C, H, W):
    """gv only / gh only equal the combined call bit for bit; grad_input (through the [B,51,H,W] kernel on converted taps)
    matches the NCHW grad_input within its run-to-run bound (its tile flush adds with atomics)."""
    inp, v, h, g = _cuda(*cases.sepconv_inputs(B, C, H, W, seed=900 + H, kind="unit"))
    gi_t, gv_t, gh_t = _tiled_grads(inp, v, h, g)
    _, gv_only, _ = _tiled_grads(inp, v, h, g, want=(False, True, False))
    _, _, gh_only = _tiled_grads(inp, v, h, g, want=(False, False, True))
    assert torch.equal(gv_only, gv_t) and torch.equal(gh_only, gh_t)
    gi_only, _, _ = _tiled_grads(inp, v, h, g, want=(True, False, False))
    gi, _, _ = _nchw_grads(inp, v, h, g, need_input=True)
    scale = float(gi.abs().max())
    for got in (gi_t, gi_only):
        assert float((got - gi).abs().max()) <= 8 * 1.1920929e-07 * scale


@pytest.mark.parametrize("B,H,W", [(1, 96, 100), (2, 64, 64), (1, 13, 21)])
def test_gray_shortcut(B, H, W):
    """Identical channel planes: one one-plane launch with the channel-summed gradient, t = (sum_c g_c) * in_0."""
    inp, v, h, g = cases.sepconv_inputs(B, 3, H, W, seed=1100 + H, kind="randn")
    inp[:, 1:] = inp[:, :1]
    ti, tv, th, tg = _cuda(inp, v, h, g)
    _, gv_gray, gh_gray = _tiled_grads(ti, tv, th, tg, gray=True, want=(False, True, True))
    _, gv_gen, gh_gen = _tiled_grads(ti, tv, th, tg, want=(False, True, True))
    for a, b in ((gv_gray, gv_gen), (gh_gray, gh_gen)):
        assert float((a - b).abs().max()) <= 2e-5 * max(1.0, float(b.abs().max()))
    gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
    _check_p(pkg.taps_from_tiled(gv_gray, H, W).cpu().numpy(), oracle.sepconv_grad_vertical_reforder(g, inp, h), gv64, "gray gv")
    _check_p(pkg.taps_from_tiled(gh_gray, H, W).cpu().numpy(), oracle.sepconv_grad_horizontal_reforder(g, inp, v), gh64, "gray gh")
    pad = _padding_mask(B, H, W)
    assert bool((gv_gray[pad] == 0).all()) and bool((gh_gray[pad] == 0).all())
    # through autograd with set_gray_replicated("assert"): the forward's decision is reused by the backward
    pkg.set_gray_replicated("assert")
    try:
        vt = pkg.taps_to_tiled(tv).requires_grad_(True)
        ht = pkg.taps_to_tiled(th).requires_grad_(True)
        pkg.SeparableConvolutionTiled.apply(ti, vt, ht).backward(tg)
    finally:
        pkg.set_gray_replicated("off")
    assert torch.equal(vt.grad, gv_gray) and torch.equal(ht.grad, gh_gray)


@pytest.mark.parametrize("B,C,H,W,bitwise", [(4, 3, 512, 512, True), (1, 3, 1001, 1004, True), (1, 3, 20, 30, False),
                                             (2, 1, 12, 13, False)])
def test_autograd_function_matches_separable_convolution(B, C, H, W, bitwise):
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(H + W)
    inp = torch.rand((B, C, H + 50, W + 50), device=dev, generator=gen)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    g = torch.randn((B, C, H, W), device=dev, generator=gen)
    vt = pkg.taps_to_tiled(v).requires_grad_(True)
    ht = pkg.taps_to_tiled(h).requires_grad_(True)
    out = pkg.SeparableConvolutionTiled.apply(inp, vt, ht)
    out.backward(g)
    _, gv, gh = _nchw_grads(inp, v, h, g)
    fwd = pkg.SeparableConvolution.apply(inp, v, h)
    assert torch.equal(out.detach(), fwd) if bitwise else float((out.detach() - fwd).abs().max()) <= 2e-6
    for got, want in ((vt.grad, pkg.taps_to_tiled(gv)), (ht.grad, pkg.taps_to_tiled(gh))):
        if bitwise:
            assert torch.equal(got, want)
        else:
            assert float((got - want).abs().max()) <= TOL * max(1.0, float(want.abs().max()))


def test_autograd_function_honours_needs_input_grad():
    B, C, H, W = 1, 3, 24, 28
    inp, v, h, g = _cuda(*cases.sepconv_inputs(B, C, H, W, seed=77, kind="unit"))
    vt, ht = pkg.taps_to_tiled(v), pkg.taps_to_tiled(h)
    gi_all, gv_all, gh_all = _tiled_grads(inp, v, h, g)
    for need in ((True, False, False), (False, True, False), (False, False, True), (True, True, False)):
        a, b, c = (t.clone().requires_grad_(n) for t, n in zip((inp, vt, ht), need))
        pkg.SeparableConvolutionTiled.apply(a, b, c).backward(g)
        for t, n, want in zip((a, b, c), need, (gi_all, gv_all, gh_all)):
            assert (t.grad is not None) == n
            if n and t is not a:
                assert torch.equal(t.grad, want)
            elif n:
                assert float((t.grad - want).abs().max()) <= 8 * 1.1920929e-07 * float(want.abs().max())


def _tail_inputs(B, C, H, W, gray, seed, dev="cuda"):
    gen = torch.Generator(device=dev).manual_seed(seed)
    i1 = torch.rand((B, C, H, W), device=dev, generator=gen)
    i2 = torch.rand((B, C, H, W), device=dev, generator=gen)
    if gray:
        i1[:, 1:] = i1[:, :1]
        i2[:, 1:] = i2[:, :1]
    taps = [torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1) for _ in range(4)]
    g = torch.rand((B, 1, H, W), device=dev, generator=gen) - 0.5
    return i1, i2, taps, g


@pytest.mark.parametrize("B,C,H,W,gray", [(1, 3, 40, 52, False), (2, 3, 37, 53, False), (1, 3, 40, 72, True), (1, 1, 24, 40, False),
                                          (1, 3, 1024, 1024, False), (1, 3, 1024, 1024, True)])
def test_tiled_interpolation_tail_gradients(B, C, H, W, gray):
    """ModuleInterpolationTailTiled: the four tap gradients, tile-major, against the fused NCHW tail and the fp64 oracle of
    the unfused expression (on a crop at 1024^2: a tap gradient only depends on its pixel's window)."""
    i1, i2, taps, g = _tail_inputs(B, C, H, W, gray, seed=H + W + C)
    tiled = [pkg.taps_to_tiled(t).requires_grad_(True) for t in taps]
    nchw = [t.clone().requires_grad_(True) for t in taps]
    pkg.set_gray_replicated("assert" if gray else "off")
    try:
        out = pkg.ModuleInterpolationTailTiled()(i1, i2, *tiled)
        fused = pkg.interpolation_tail(i1, i2, *nchw)
        assert torch.equal(out.detach(), pkg.interpolation_tail_tiled(i1, i2, *(t.detach() for t in tiled)))
    finally:
        pkg.set_gray_replicated("off")
    out.backward(g)
    fused.backward(g)
    pad = _padding_mask(B, H, W)
    for t, n in zip(tiled, nchw):
        assert float((pkg.taps_from_tiled(t.grad, H, W) - n.grad).abs().max()) <= 4e-6
        assert bool((t.grad[pad] == 0).all())
    if H * W <= 4096:
        want = oracle.interp_tail_grads_f64(*(x.cpu().numpy() for x in (g, i1, i2, *taps)))
        got = [pkg.taps_from_tiled(t.grad, H, W).cpu().numpy() for t in tiled]
    else:
        y0, x0, hh, ww = 500, 300, 16, 24
        gc = np.repeat(g[:, :, y0:y0 + hh, x0:x0 + ww].cpu().numpy() / np.float32(C), C, axis=1)
        want = []
        for f, (kv, kh) in ((i1, taps[:2]), (i2, taps[2:])):
            fc = f[:, :, y0 - 25:y0 + hh + 25, x0 - 25:x0 + ww + 25].cpu().numpy()
            want += oracle.sepconv_grad_taps_f64(gc, fc, *(k[:, :, y0:y0 + hh, x0:x0 + ww].cpu().numpy().copy() for k in (kv, kh)))
        got = [pkg.taps_from_tiled(t.grad, H, W)[:, :, y0:y0 + hh, x0:x0 + ww].cpu().numpy() for t in tiled]
    for a, b in zip(got, want):
        assert np.abs(a - b).max() <= TOL * max(1.0, float(np.abs(b).max()))


def test_tiled_tail_refuses_frame_gradients():
    i1, i2, taps, g = _tail_inputs(1, 3, 16, 16, False, seed=5)
    tiled = [pkg.taps_to_tiled(t).requires_grad_(True) for t in taps]
    out = pkg.ModuleInterpolationTailTiled()(i1.requires_grad_(True), i2, *tiled)
    with pytest.raises(NotImplementedError):
        out.backward(g)


@pytest.mark.parametrize("C,H,W", [(3, 37, 45), (1, 20, 29), (3, 512, 508)])
def test_inf_in_the_last_input_column_leaves_the_padding_zero(C, H, W):
    """Padding entries are stored as zeros, not as sum g * P: g is zero there, but P reaches real input columns W..W+49."""
    inp, v, h, g = _cuda(*cases.sepconv_inputs(1, C, H, W, seed=31 + C, kind="unit"))
    inp[:, :, :, -1] = float("inf")
    for gray in ((False, True) if C == 3 else (False,)):
        _, gv_t, gh_t = _tiled_grads(inp, v, h, g, gray=gray, want=(False, True, True))
        pad = _padding_mask(1, H, W)
        assert bool((gv_t[pad] == 0).all()) and bool((gh_t[pad] == 0).all())
        inner = pkg.taps_from_tiled(gv_t, H, W)[:, :, :, : W - 1]      # pixels whose window stops short of the Inf column
        assert bool(torch.isfinite(inner).all())


def test_run_to_run_determinism_with_one_hot_taps():
    """The shared-memory tap buffers are refilled by TMA while other warps' loads are queued (the refill-overtakes-load
    hazard of DESIGN 4.1): with one-hot taps a single wrong tap value changes the result visibly."""
    dev = "cuda"
    B, C, H, W = 2, 3, 512, 512
    torch.manual_seed(11)
    x = torch.rand((B, C, H + 50, W + 50), device=dev)
    gen = torch.Generator(device="cpu").manual_seed(29)
    fy = torch.randint(0, 51, (B, 1, H, W), generator=gen).to(dev)
    fx = torch.randint(0, 51, (B, 1, H, W), generator=gen).to(dev)
    v = torch.zeros((B, 51, H, W), device=dev).scatter_(1, fy, 1.0)
    h = torch.zeros((B, 51, H, W), device=dev).scatter_(1, fx, 1.0)
    g = torch.randn((B, C, H, W), device=dev)
    ref = _tiled_grads(x, v, h, g, want=(False, True, True))
    for _ in range(2):
        cur = _tiled_grads(x, v, h, g, want=(False, True, True))
        assert torch.equal(cur[1], ref[1]) and torch.equal(cur[2], ref[2])
