"""GPU parity tests for the sepconv path.  Everything goes through the C ABI (via the
reference-shaped autograd Function); the oracle is only the checker.

Tolerances (SURVEY.md section 8c):
  P0  CPU oracle (reference order) vs the reference's own .cu on the B200: bit-equal.
  P1  unit-scale inputs (|out| <~ 1): max-abs <= 1e-5 vs the reference-order oracle.
  P2  raw N(0,1) taps (|out| up to ~1e2): max-abs <= 1e-5 * max(1, max|ref|) AND the
      kernel's error vs fp64 does not exceed the reference order's own error.
  STRICT_ORDER flag: bit-equal to the reference order.
"""
import os

import numpy as np
import pytest
import torch

import oracle
from tests.golden import cases

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _cuda(*arrs):
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs)


def _ops():
    import sstem_restoration_b200 as pkg
    return pkg


def _fwd(inp, v, h, strict=False):
    pkg = _ops()
    pkg.set_strict_order(strict)
    try:
        return pkg.SeparableConvolution.apply(inp, v, h)
    finally:
        pkg.set_strict_order(False)


def _bwd(inp, v, h, g, need_input=True):
    pkg = _ops()
    inp = inp.clone().requires_grad_(need_input)
    v = v.clone().requires_grad_(True)
    h = h.clone().requires_grad_(True)
    out = pkg.SeparableConvolution.apply(inp, v, h)
    out.backward(g)
    return out.detach(), inp.grad, v.grad, h.grad


def _check_p(got, ref32, ref64, what):
    scale = max(1.0, float(np.abs(ref64).max()))
    err_vs_ref = float(np.abs(got.astype(np.float64) - ref32).max())
    err_new = float(np.abs(got - ref64).max())
    err_ref = float(np.abs(ref32 - ref64).max())
    assert err_vs_ref <= TOL * scale, f"{what}: |new-ref|={err_vs_ref:.3e} scale={scale:.3g}"
    assert err_new <= max(err_ref * 1.25, 2e-6 * scale), f"{what}: err(new,f64)={err_new:.3e} > err(ref,f64)={err_ref:.3e}"


# ---------------------------------------------------------------- P0: pin the oracle
@pytest.mark.parametrize("name", [n for n, p in cases.sepconv_cases().items() if p["C"] == 3])
def test_p0_oracle_equals_reference_cuda(name, golden_dir):
    """The reference's outputs: its own .cu compiled verbatim for sm_100a and run on a B200 (sepconv_ref.npz)."""
    inp, v, h, g = cases.sepconv_inputs(**cases.sepconv_cases()[name])
    ref = np.load(os.path.join(golden_dir, "sepconv_ref.npz"))
    out, gi, gv, gh = (ref[name + s] for s in ("_out", "_gi", "_gv", "_gh"))
    assert np.array_equal(out.view(np.uint32), oracle.sepconv_forward_reforder(inp, v, h).view(np.uint32))
    assert np.array_equal(gv.view(np.uint32), oracle.sepconv_grad_vertical_reforder(g, inp, h).view(np.uint32))
    assert np.array_equal(gh.view(np.uint32), oracle.sepconv_grad_horizontal_reforder(g, inp, v).view(np.uint32))
    assert not gi.any()   # SeparableConvolution.py:60 -- the reference never computes it


def test_golden_fixture_matches_kernel_strict(golden_dir):
    path = os.path.join(golden_dir, "sepconv_ref.npz")
    if not os.path.exists(path):
        pytest.skip("sepconv_ref.npz not committed yet")
    ref = np.load(path)
    for name, p in cases.sepconv_cases().items():
        if p["C"] != 3:
            continue
        inp, v, h, g = cases.sepconv_inputs(**p)
        got = _fwd(*_cuda(inp, v, h), strict=True).cpu().numpy()
        assert np.array_equal(got.view(np.uint32), ref[name + "_out"].view(np.uint32)), name


# ---------------------------------------------------------------- forward
@pytest.mark.parametrize("name", list(cases.sepconv_cases()))
def test_forward_strict_order_is_bit_exact(name):
    inp, v, h, g = cases.sepconv_inputs(**cases.sepconv_cases()[name])
    got = _fwd(*_cuda(inp, v, h), strict=True).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), oracle.sepconv_forward_reforder(inp, v, h).view(np.uint32))


@pytest.mark.parametrize("name", list(cases.sepconv_cases()))
def test_forward_parity(name):
    inp, v, h, g = cases.sepconv_inputs(**cases.sepconv_cases()[name])
    got = _fwd(*_cuda(inp, v, h)).cpu().numpy()
    _check_p(got, oracle.sepconv_forward_reforder(inp, v, h), oracle.sepconv_forward_f64(inp, v, h), "fwd " + name)


@pytest.mark.parametrize("B,C,H,W", [(1, 3, 1, 1), (1, 1, 1, 70), (1, 3, 70, 1), (2, 2, 33, 65), (1, 4, 8, 129),
                                      (3, 3, 17, 31), (1, 3, 64, 64), (1, 1, 40, 200), (1, 5, 9, 9)])
def test_forward_ragged_shapes(B, C, H, W):
    inp, v, h, g = cases.sepconv_inputs(B, C, H, W, seed=1000 + H * W + C, kind="unit")
    got = _fwd(*_cuda(inp, v, h)).cpu().numpy()
    _check_p(got, oracle.sepconv_forward_reforder(inp, v, h), oracle.sepconv_forward_f64(inp, v, h), f"fwd {B,C,H,W}")


# ---------------------------------------------------------------- backward
@pytest.mark.parametrize("name", list(cases.sepconv_cases()))
def test_backward_parity(name):
    p = cases.sepconv_cases()[name]
    inp, v, h, g = cases.sepconv_inputs(**p)
    out, gi, gv, gh = _bwd(*_cuda(inp, v, h, g))
    gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
    _check_p(gv.cpu().numpy(), oracle.sepconv_grad_vertical_reforder(g, inp, h), gv64, "gv " + name)
    _check_p(gh.cpu().numpy(), oracle.sepconv_grad_horizontal_reforder(g, inp, v), gh64, "gh " + name)
    gi64 = oracle.sepconv_grad_input_f64(g, v, h)
    scale = max(1.0, float(np.abs(gi64).max()))
    assert np.abs(gi.cpu().numpy() - gi64).max() <= TOL * scale, "gi " + name


@pytest.mark.parametrize("B,C,H,W", [(1, 3, 1, 1), (1, 1, 5, 70), (2, 2, 33, 37), (1, 4, 8, 66), (1, 3, 64, 64), (2, 3, 19, 130)])
def test_backward_ragged_shapes(B, C, H, W):
    inp, v, h, g = cases.sepconv_inputs(B, C, H, W, seed=2000 + H * W + C, kind="unit")
    out, gi, gv, gh = _bwd(*_cuda(inp, v, h, g))
    gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
    _check_p(gv.cpu().numpy(), oracle.sepconv_grad_vertical_reforder(g, inp, h), gv64, f"gv {B,C,H,W}")
    _check_p(gh.cpu().numpy(), oracle.sepconv_grad_horizontal_reforder(g, inp, v), gh64, f"gh {B,C,H,W}")
    gi64 = oracle.sepconv_grad_input_f64(g, v, h)
    assert np.abs(gi.cpu().numpy() - gi64).max() <= TOL * max(1.0, float(np.abs(gi64).max()))


def test_needs_input_grad_is_honoured():
    inp, v, h, g = _cuda(*cases.sepconv_inputs(1, 3, 8, 8, seed=5, kind="unit"))
    out, gi, gv, gh = _bwd(inp, v, h, g, need_input=False)
    assert gi is None and gv is not None and gh is not None
    pkg = _ops()
    v2 = v.clone().requires_grad_(True)
    pkg.SeparableConvolution.apply(inp, v2, h).backward(g)
    assert torch.equal(v2.grad, gv)


def test_reference_gradcheck_recipe():
    """sff_scripts_interp/model/model_interp.py:109-119: randn(2,3,51,51), taps (2,51,1,1), eps=atol=rtol=1e-2."""
    torch.manual_seed(0)
    pkg = _ops()
    inputs = (torch.randn(2, 3, 51, 51, device="cuda"),
              torch.randn(2, 51, 1, 1, device="cuda", requires_grad=True),
              torch.randn(2, 51, 1, 1, device="cuda", requires_grad=True))
    assert torch.autograd.gradcheck(pkg.SeparableConvolution.apply, inputs, eps=1e-2, atol=1e-2, rtol=1e-2,
                                    nondet_tol=0.0, check_grad_dtypes=False)


def test_gradcheck_including_input():
    torch.manual_seed(1)
    pkg = _ops()
    inputs = (torch.randn(1, 2, 53, 52, device="cuda", requires_grad=True),
              torch.randn(1, 51, 3, 2, device="cuda", requires_grad=True),
              torch.randn(1, 51, 3, 2, device="cuda", requires_grad=True))
    assert torch.autograd.gradcheck(pkg.SeparableConvolution.apply, inputs, eps=1e-2, atol=2e-2, rtol=2e-2,
                                    check_grad_dtypes=False)


# ---------------------------------------------------------------- generic tap counts (CuPy-variant surface)
@pytest.mark.parametrize("K", [1, 5, 13, 33, 64])
def test_function_sepconv_generic_taps(K):
    pkg = _ops()
    r = np.random.default_rng(K)
    B, C, H, W = 2, 3, 11, 14
    inp = r.standard_normal((B, C, H + K - 1, W + K - 1)).astype(np.float32)
    v = (r.standard_normal((B, K, H, W)) / K).astype(np.float32)
    h = (r.standard_normal((B, K, H, W))).astype(np.float32)
    g = r.standard_normal((B, C, H, W)).astype(np.float32)
    ti, tv, th, tg = _cuda(inp, v, h, g)
    ti.requires_grad_(True); tv.requires_grad_(True); th.requires_grad_(True)
    out = pkg.FunctionSepconv(ti, tv, th)
    out.backward(tg)
    ref64 = oracle.sepconv_forward_f64(inp, v, h)
    assert np.abs(out.detach().cpu().numpy() - ref64).max() <= TOL * max(1.0, np.abs(ref64).max())
    gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
    gi64 = oracle.sepconv_grad_input_f64(g, v, h)
    for got, ref in ((tv.grad, gv64), (th.grad, gh64), (ti.grad, gi64)):
        assert np.abs(got.cpu().numpy() - ref).max() <= TOL * max(1.0, np.abs(ref).max())
    out2 = pkg.ModuleSepconv()(ti.detach(), tv.detach(), th.detach())
    assert torch.equal(out2, out.detach())


# ---------------------------------------------------------------- full-size, size-independent properties
def _one_hot_taps(B, H, W, seed, device):
    gen = torch.Generator(device="cpu").manual_seed(seed)
    fy = torch.randint(0, 51, (B, 1, H, W), generator=gen).to(device)
    fx = torch.randint(0, 51, (B, 1, H, W), generator=gen).to(device)
    v = torch.zeros((B, 51, H, W), device=device).scatter_(1, fy, 1.0)
    h = torch.zeros((B, 51, H, W), device=device).scatter_(1, fx, 1.0)
    return fy, fx, v, h


@pytest.mark.parametrize("B,C,H,W", [(1, 3, 256, 256), (2, 3, 512, 512), (1, 3, 2048, 2048), (1, 1, 1000, 1500)])
def test_one_hot_taps_select_exact_pixels_at_full_size(B, C, H, W):
    """With one-hot v and h the op is a pure gather: out[b,c,y,x] = in[b,c,y+fy,x+fx] EXACTLY."""
    dev = "cuda"
    torch.manual_seed(3)
    inp = torch.rand((B, C, H + 50, W + 50), device=dev)
    fy, fx, v, h = _one_hot_taps(B, H, W, 17, dev)
    out = _fwd(inp, v, h)
    yy = torch.arange(H, device=dev).view(1, 1, H, 1) + fy
    xx = torch.arange(W, device=dev).view(1, 1, 1, W) + fx
    flat = (yy * (W + 50) + xx).expand(B, C, H, W).reshape(B, C, -1)
    expect = inp.reshape(B, C, -1).gather(2, flat).reshape(B, C, H, W)
    assert torch.equal(out, expect)
    del v, h
    torch.cuda.empty_cache()


def test_linearity_and_tap_gradients_at_training_size():
    """C3-sized slice: linear in the input; with one-hot taps the tap gradients are plain
    channel sums of g * shifted input (checked against torch within fp32 rounding of a C-term sum)."""
    dev = "cuda"
    B, C, H, W = 2, 3, 512, 512
    torch.manual_seed(4)
    x1 = torch.rand((B, C, H + 50, W + 50), device=dev)
    x2 = torch.rand((B, C, H + 50, W + 50), device=dev)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    a = 0.5
    lhs = _fwd(a * x1 + x2, v, h)
    rhs = a * _fwd(x1, v, h) + _fwd(x2, v, h)
    assert (lhs - rhs).abs().max().item() <= 1e-5
    fy, fx, v1, h1 = _one_hot_taps(B, H, W, 23, dev)
    g = torch.randn((B, C, H, W), device=dev)
    out, gi, gv, gh = _bwd(x1, v1, h1, g, need_input=False)
    # gv[b,f,y,x] = sum_c g * in[b,c,y+f,x+fx]
    for f in (0, 25, 50):
        yy = torch.arange(H, device=dev).view(1, 1, H, 1) + f
        xx = torch.arange(W, device=dev).view(1, 1, 1, W) + fx
        flat = (yy * (W + 50) + xx).expand(B, C, H, W).reshape(B, C, -1)
        exp_v = (g * x1.reshape(B, C, -1).gather(2, flat).reshape(B, C, H, W)).sum(1)
        assert (gv[:, f] - exp_v).abs().max().item() <= 1e-5
        yy = torch.arange(H, device=dev).view(1, 1, H, 1) + fy
        xx = torch.arange(W, device=dev).view(1, 1, 1, W) + f
        flat = (yy * (W + 50) + xx).expand(B, C, H, W).reshape(B, C, -1)
        exp_h = (g * x1.reshape(B, C, -1).gather(2, flat).reshape(B, C, H, W)).sum(1)
        assert (gh[:, f] - exp_h).abs().max().item() <= 1e-5


def test_adjoint_identity_for_grad_input():
    """<sepconv(x), g> == <x, grad_input(g)>: ties the computed grad_input to the forward at a mid size."""
    dev = "cuda"
    B, C, H, W = 1, 3, 96, 160
    torch.manual_seed(5)
    x = torch.randn((B, C, H + 50, W + 50), device=dev)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    g = torch.randn((B, C, H, W), device=dev)
    out, gi, gv, gh = _bwd(x, v, h, g)
    lhs = (out.double() * g.double()).sum().item()
    rhs = (x.double() * gi.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))


def test_other_device_stream_and_noncurrent_stream():
    """Calls are stream-ordered on torch's current stream."""
    inp, v, h, g = _cuda(*cases.sepconv_inputs(1, 3, 32, 32, seed=9, kind="unit"))
    ref = _fwd(inp, v, h)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = _fwd(inp, v, h)
    s.synchronize()
    assert torch.equal(ref, got)


def test_host_buffer_pipeline_matches_device_path():
    """sepconv_forward_backward_host (chunked, multi-stream, pinned buffers) == the autograd op."""
    pkg = _ops()
    inp, v, h, g = cases.sepconv_inputs(5, 3, 24, 40, seed=77, kind="unit")
    ti, tv, th, tg = (torch.from_numpy(a) for a in (inp, v, h, g))
    out, gv, gh = pkg.sepconv_forward_backward_host(ti.pin_memory(), tv.pin_memory(), th.pin_memory(), tg.pin_memory(), chunk=2)
    # no synchronize here: with join=True (default) the pinned results are complete when the call returns
    got = (out.clone(), gv.clone(), gh.clone())
    ref_out, _, ref_gv, ref_gh = _bwd(*_cuda(inp, v, h, g), need_input=False)
    assert torch.equal(got[0], ref_out.cpu()) and torch.equal(got[1], ref_gv.cpu()) and torch.equal(got[2], ref_gh.cpu())
    only = pkg.sepconv_forward_backward_host(ti, tv, th).clone()  # forward only, pageable memory
    assert torch.equal(only, ref_out.cpu())


def test_gray_replicated_shortcut():
    """SSTEM_SEPCONV_GRAY_REPLICATED: identical channel planes (the reference's gray x3 inputs).
    Forward bit-identical to the general path; tap gradients within tolerance of fp64."""
    pkg = _ops()
    r = np.random.default_rng(5)
    B, H, W = 2, 21, 45
    plane = r.random((B, 1, H + 50, W + 50), dtype=np.float32)
    inp = np.repeat(plane, 3, axis=1)
    _, v, h, g = cases.sepconv_inputs(B, 3, H, W, seed=6, kind="unit")
    ti, tv, th, tg = _cuda(inp, v, h, g)
    ref_out, _, ref_gv, ref_gh = _bwd(ti, tv, th, tg, need_input=False)
    for mode in ("assert", "detect"):
        pkg.set_gray_replicated(mode)
        try:
            out, _, gv, gh = _bwd(ti, tv, th, tg, need_input=False)
        finally:
            pkg.set_gray_replicated("off")
        assert torch.equal(out, ref_out), mode
        gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
        _check_p(gv.cpu().numpy(), oracle.sepconv_grad_vertical_reforder(g, inp, h), gv64, "gray gv " + mode)
        _check_p(gh.cpu().numpy(), oracle.sepconv_grad_horizontal_reforder(g, inp, v), gh64, "gray gh " + mode)
    # detection must NOT fire on planes that differ
    inp2 = inp.copy(); inp2[0, 1, 3, 3] += 0.5
    t2 = torch.from_numpy(inp2).cuda()
    pkg.set_gray_replicated("detect")
    try:
        out2 = pkg.SeparableConvolution.apply(t2, tv, th)
    finally:
        pkg.set_gray_replicated("off")
    assert torch.equal(out2, pkg.SeparableConvolution.apply(t2, tv, th))


def test_gray_detection_on_the_device_at_training_size():
    """"detect" / "auto": the planes are compared by a kernel, both paths are launched gated on a DEVICE flag (no host sync).
    The flag must say gray exactly when the planes are identical, the forward must be bit-identical to the general path both
    ways, and the tap gradients must agree with the general path's to fp32 rounding."""
    from sstem_restoration_b200 import _lib
    pkg = _ops()
    dev = "cuda"
    B, H, W = 2, 512, 512
    gen = torch.Generator(device=dev).manual_seed(21)
    plane = torch.rand((B, 1, H + 50, W + 50), device=dev, generator=gen)
    gray = plane.expand(B, 3, H + 50, W + 50).contiguous()
    color = gray.clone()
    color[1, 2, 300, 17] += 0.25                                  # one differing element in the last image
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev, generator=gen), 1)
    g = torch.randn((B, 3, H, W), device=dev, generator=gen)
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    for inp, want in ((gray, True), (color, False)):
        pkg.set_gray_replicated("off")
        ref_out, _, ref_gv, ref_gh = _bwd(inp, v, h, g, need_input=False)
        flag = torch.full((1,), 77, dtype=torch.int32, device=dev)
        out = torch.empty_like(ref_out)
        assert lib.sstem_sepconv_forward_detect(inp.data_ptr(), v.data_ptr(), h.data_ptr(), out.data_ptr(), B, 3, H, W, 51, 0,
                                                flag.data_ptr(), st) == 0
        assert (int(flag.item()) != 0) == want and torch.equal(out, ref_out)
        for mode in ("detect", "auto"):
            pkg.set_gray_replicated(mode)
            try:
                out2, _, gv, gh = _bwd(inp, v, h, g, need_input=False)
            finally:
                pkg.set_gray_replicated("off")
            assert torch.equal(out2, ref_out), mode
            tol = 2e-5 * max(1.0, float(ref_gv.abs().max()), float(ref_gh.abs().max()))
            assert float((gv - ref_gv).abs().max()) <= tol and float((gh - ref_gh).abs().max()) <= tol, mode
            if not want:                                          # planes differ: the general path ran, bit for bit
                assert torch.equal(gv, ref_gv) and torch.equal(gh, ref_gh)


def test_window_rows_outside_a_pixels_support_cannot_leak_nan():
    """The tuned kernels walk 58 input rows per 8-row tile; a row below a pixel's own 51-row window
    is multiplied by a zero weight internally.  A NaN / Inf there must not reach that pixel."""
    pkg = _ops()
    inp, v, h, g = cases.sepconv_inputs(1, 3, 8, 40, seed=12, kind="unit")
    ref = _fwd(*_cuda(inp, v, h)).cpu().numpy()
    bad = inp.copy()
    bad[:, :, 57, :] = np.nan            # last input row: only output row 7 may see it
    bad[:, :, 56, 5] = np.inf            # row 56: only output rows 6, 7
    got = _fwd(*_cuda(bad, v, h)).cpu().numpy()
    assert np.array_equal(got[:, :, :6], ref[:, :, :6])          # rows 0..5 untouched, bit for bit
    assert np.isnan(got[:, :, 7]).all()
    out, gi, gv, gh = _bwd(*_cuda(bad, v, h, g), need_input=False)
    assert torch.isfinite(gv[:, :, :6]).all() and torch.isfinite(gh[:, :, :6]).all()


def test_operator_runs_on_a_non_current_device_stream_pair():
    """Replica-thread pattern (nn.DataParallel): tensors decide the device, not the caller's context."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    pkg = _ops()
    inp, v, h, g = cases.sepconv_inputs(1, 3, 16, 16, seed=13, kind="unit")
    ref = _fwd(*_cuda(inp, v, h)).cpu()
    t = [torch.from_numpy(a).to("cuda:1") for a in (inp, v, h)]
    assert torch.cuda.current_device() == 0
    out = pkg.SeparableConvolution.apply(*t)
    assert out.device.index == 1 and torch.equal(out.cpu(), ref)


# ---------------------------------------------------------------- BASELINE config 2: taps from the reference's own KPN
def _kpn_crop_inputs(golden_dir):
    p = cases.kpn_taps_case()
    taps = np.load(os.path.join(golden_dir, "kpn_taps_ref.npz"))
    x = cases.kpn_frames(p)
    y0, x0, n = p["crop_y"], p["crop_x"], p["crop"]
    pad = lambda f: np.pad(f, ((0, 0), (0, 0), (25, 25), (25, 25)), mode="edge")[:, :, y0:y0 + n + 50, x0:x0 + n + 50]
    return np.ascontiguousarray(pad(x[:, :3])), np.ascontiguousarray(pad(x[:, 3:6])), taps


def test_c2_taps_from_reference_kpn(golden_dir):
    """Raw 51-tap kernels predicted by the reference's random-init IFNet (tests/golden/make_kpn_taps_golden.py; |taps| up
    to ~6, |out| ~ 1e1): protocol P2 for the forward of both frames and for the tap gradients."""
    i1, i2, taps = _kpn_crop_inputs(golden_dir)
    g = np.random.default_rng(5).standard_normal((1, 3, 32, 32)).astype(np.float32)
    for inp, v, h in ((i2, taps["k2v"], taps["k2h"]), (i1, taps["k1v"], taps["k1h"])):
        out, gi, gv, gh = _bwd(*_cuda(inp, v, h, g), need_input=False)
        _check_p(out.cpu().numpy(), oracle.sepconv_forward_reforder(inp, v, h), oracle.sepconv_forward_f64(inp, v, h), "kpn fwd")
        gv64, gh64 = oracle.sepconv_grad_taps_f64(g, inp, v, h)
        _check_p(gv.cpu().numpy(), oracle.sepconv_grad_vertical_reforder(g, inp, h), gv64, "kpn gv")
        _check_p(gh.cpu().numpy(), oracle.sepconv_grad_horizontal_reforder(g, inp, v), gh64, "kpn gh")
        strict = _fwd(*_cuda(inp, v, h), strict=True).cpu().numpy()
        assert np.array_equal(strict.view(np.uint32), oracle.sepconv_forward_reforder(inp, v, h).view(np.uint32))


def test_persistent_kernels_are_run_to_run_deterministic():
    """The persistent (third-generation) kernels refill their shared-memory tap buffers with TMA while other warps keep
    the shared-memory pipe busy; a refill that overtakes queued loads shows up as a few wrong pixels that differ from run
    to run (it did, once).  Forward, grad_vertical and grad_horizontal must be bit-identical over repeated launches."""
    dev = "cuda"
    B, C, H, W = 2, 3, 512, 512
    torch.manual_seed(11)
    x = torch.rand((B, C, H + 50, W + 50), device=dev)
    fy, fx, v0, h0 = _one_hot_taps(B, H, W, 29, dev)        # one-hot taps: a single wrong tap value changes the result visibly
    g = torch.randn((B, C, H, W), device=dev)
    ref = None
    for _ in range(12):
        out, _, gv, gh = _bwd(x, v0, h0, g, need_input=False)
        cur = (out, gv, gh)
        if ref is None:
            ref = cur
        else:
            for a, b, name in zip(ref, cur, ("out", "grad_vertical", "grad_horizontal")):
                assert torch.equal(a, b), f"{name} differs between two launches on identical inputs"


@pytest.mark.parametrize("B,H,W", [(1, 1001, 1004), (3, 509, 516)])
def test_persistent_kernels_on_ragged_large_shapes(B, H, W):
    """Sizes that take the persistent kernels but are no multiple of their tiles (8 rows / 32 columns; the last CTA tile has
    partially and fully out-of-image warp tiles): one-hot taps make the forward an exact gather and the tap gradients
    plain channel sums of g * shifted input."""
    dev = "cuda"
    C = 3
    torch.manual_seed(6)
    x = torch.rand((B, C, H + 50, W + 50), device=dev)
    fy, fx, v1, h1 = _one_hot_taps(B, H, W, 31, dev)
    g = torch.randn((B, C, H, W), device=dev)
    out, _, gv, gh = _bwd(x, v1, h1, g, need_input=False)
    yy = torch.arange(H, device=dev).view(1, 1, H, 1) + fy
    xx = torch.arange(W, device=dev).view(1, 1, 1, W) + fx
    flat = (yy * (W + 50) + xx).expand(B, C, H, W).reshape(B, C, -1)
    assert torch.equal(out, x.reshape(B, C, -1).gather(2, flat).reshape(B, C, H, W))
    for f in (0, 17, 50):
        yy = torch.arange(H, device=dev).view(1, 1, H, 1) + f
        flat = (yy * (W + 50) + (torch.arange(W, device=dev).view(1, 1, 1, W) + fx)).expand(B, C, H, W).reshape(B, C, -1)
        exp_v = (g * x.reshape(B, C, -1).gather(2, flat).reshape(B, C, H, W)).sum(1)
        assert (gv[:, f] - exp_v).abs().max().item() <= 1e-5
        flat = ((torch.arange(H, device=dev).view(1, 1, H, 1) + fy) * (W + 50) + torch.arange(W, device=dev).view(1, 1, 1, W) + f).expand(B, C, H, W).reshape(B, C, -1)
        exp_h = (g * x.reshape(B, C, -1).gather(2, flat).reshape(B, C, H, W)).sum(1)
        assert (gh[:, f] - exp_h).abs().max().item() <= 1e-5
    # untouched guard band: the kernels must not write outside [B,51,H,W] / [B,C,H,W] (checked by the allocator's neighbours
    # indirectly; here: a second run gives identical bits)
    out2, _, gv2, gh2 = _bwd(x, v1, h1, g, need_input=False)
    assert torch.equal(out, out2) and torch.equal(gv, gv2) and torch.equal(gh, gh2)


def test_grad_input_run_to_run_bound_and_nan_footprint():
    """grad_input's tile flush uses global atomic adds (up to ~14 tiles overlap on an element), so the summation ORDER may
    differ between launches: pin the bound (a few ulps of the largest partial sum) instead of pretending bit-determinism, and
    check that a NaN in the upstream gradient reaches exactly its 51 x 51 footprint (the flush skips exact zeros only)."""
    dev = "cuda"
    B, C, H, W = 1, 3, 96, 128
    torch.manual_seed(15)
    x = torch.rand((B, C, H + 50, W + 50), device=dev)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    g = torch.randn((B, C, H, W), device=dev)
    runs = [_bwd(x, v, h, g)[1] for _ in range(4)]
    scale = float(runs[0].abs().max())
    worst = max(float((r - runs[0]).abs().max()) for r in runs[1:])
    assert worst <= 8 * 1.1920929e-07 * scale, f"run-to-run spread {worst:.3e} at scale {scale:.3g}"
    g2 = g.clone()
    g2[0, 1, 40, 70] = float("nan")
    gi = _bwd(x, v, h, g2)[1]
    nan = torch.isnan(gi)
    expect = torch.zeros_like(nan)
    expect[0, 1, 40:40 + 51, 70:70 + 51] = True
    assert torch.equal(nan, expect)
