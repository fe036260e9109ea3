"""GPU parity tests for the two warps: bit-equality with the reference's own outputs
(tests/golden/warp_*.npz, produced by importing the reference in the build container)
and with the oracle restatement on larger seeded inputs; exact properties at full size."""
import os

import numpy as np
import pytest
import torch

import oracle
from tests.golden import cases

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ---------------------------------------------------------------- SpatialTransformation
@pytest.mark.parametrize("name", list(cases.warp_torch_cases()))
@pytest.mark.parametrize("nhwc", [False, True])
def test_spatial_transformation_matches_reference_bitwise(golden_dir, name, nhwc):
    from sstem_restoration_b200 import SpatialTransformation
    ref = np.load(os.path.join(golden_dir, "warp_torch_ref.npz"))[name]
    moving, flow = cases.warp_torch_cases()[name]
    st = SpatialTransformation(use_gpu=True, nhwc_memory=nhwc)
    got = st(torch.from_numpy(moving).cuda(), torch.from_numpy(flow).cuda())
    assert tuple(got.shape) == ref.shape
    if nhwc:
        assert got.permute(0, 2, 3, 1).is_contiguous()
    assert np.array_equal(_bits(got.contiguous().cpu().numpy()), _bits(ref)), name


@pytest.mark.parametrize("name", ["b1c3_noise", "b3c3_wide", "b1c2_fold"])
def test_spatial_transformation_planar_flow_view_and_host_tensors(golden_dir, name):
    """Every reference call site passes pred_flow.permute(0,2,3,1), a strided view of planar
    [B,2,H,W] (sff_scripts_fusion/inference.py:149); host tensors round-trip through the GPU."""
    from sstem_restoration_b200 import SpatialTransformation
    ref = np.load(os.path.join(golden_dir, "warp_torch_ref.npz"))[name]
    moving, flow = cases.warp_torch_cases()[name]
    planar = torch.from_numpy(np.ascontiguousarray(flow.transpose(0, 3, 1, 2))).cuda()
    view = planar.permute(0, 2, 3, 1)
    assert not view.is_contiguous() or view.shape[1] == 1
    got = SpatialTransformation(True)(torch.from_numpy(moving).cuda(), view)
    assert np.array_equal(_bits(got.cpu().numpy()), _bits(ref))
    got_host = SpatialTransformation(False)(torch.from_numpy(moving), torch.from_numpy(flow))
    assert not got_host.is_cuda and np.array_equal(_bits(got_host.numpy()), _bits(ref))


@pytest.mark.parametrize("B,C,H,W,sigma", [(1, 3, 512, 512, 5.0), (2, 1, 300, 333, 2.0), (1, 3, 257, 1023, 40.0)])
def test_spatial_transformation_matches_oracle_bitwise(B, C, H, W, sigma):
    from sstem_restoration_b200 import SpatialTransformation
    r = np.random.default_rng(H * W)
    moving = r.random((B, C, H, W), dtype=np.float32)
    flow = (sigma * r.standard_normal((B, H, W, 2))).astype(np.float32)
    got = SpatialTransformation(True)(torch.from_numpy(moving).cuda(), torch.from_numpy(flow).cuda())
    assert np.array_equal(_bits(got.cpu().numpy()), _bits(oracle.warp_torch_restated(moving, flow)))


@pytest.mark.parametrize("H,W", [(2048, 2048), (4096, 4096)])
def test_spatial_transformation_exact_properties_at_full_size(H, W):
    """Zero flow is the identity; an integer shift is an exact shifted copy with a zero border."""
    from sstem_restoration_b200 import SpatialTransformation
    st = SpatialTransformation(True)
    torch.manual_seed(0)
    moving = torch.rand((1, 3, H, W), device="cuda")
    planar = torch.zeros((1, 2, H, W), device="cuda")
    assert torch.equal(st(moving, planar.permute(0, 2, 3, 1)), moving)
    dx, dy = 7, -3
    planar[:, 0] = dx
    planar[:, 1] = dy
    got = st(moving, planar.permute(0, 2, 3, 1))
    expect = torch.zeros_like(moving)
    expect[:, :, -dy:, : W - dx] = moving[:, :, : H + dy, dx:]
    assert torch.equal(got, expect)


def test_spatial_transformation_backward_matches_reference_autograd(golden_dir):
    """Gradients w.r.t. the moving image and the flow against autograd through the reference's own module
    (tests/golden/warp_torch_grad_ref.npz) and the oracle restatement; planar-strided flow view and NHWC memory too."""
    from sstem_restoration_b200 import SpatialTransformation
    from tests.golden.make_warp_grad_golden import upstream
    ref = np.load(os.path.join(golden_dir, "warp_torch_grad_ref.npz"))
    for name, (mv, fl) in cases.warp_torch_cases().items():
        if name + "_gm" not in ref:
            continue
        g = torch.from_numpy(upstream(name, mv.shape)).cuda()
        om, of = oracle.warp_torch_backward_restated(mv, fl, g.cpu().numpy())
        for variant in ("interleaved", "planar_view", "nhwc"):
            m = torch.from_numpy(mv).cuda().requires_grad_(True)
            if variant == "planar_view":
                base = torch.from_numpy(np.ascontiguousarray(fl.transpose(0, 3, 1, 2))).cuda().requires_grad_(True)
                f = base.permute(0, 2, 3, 1)
            else:
                base = f = torch.from_numpy(fl).cuda().requires_grad_(True)
            out = SpatialTransformation(True, nhwc_memory=(variant == "nhwc"))(m, f)
            out.backward(g)
            gf = base.grad.permute(0, 2, 3, 1) if variant == "planar_view" else base.grad
            for got, want in ((m.grad, ref[name + "_gm"]), (gf, ref[name + "_gf"]), (m.grad, om), (gf, of)):
                assert np.abs(got.cpu().numpy() - want).max() <= 2e-5 * max(1.0, np.abs(want).max()), (name, variant)


@pytest.mark.parametrize("kind", ["fold", "noise2"])
def test_spatial_transformation_backward_through_a_planar_view_at_512(kind):
    """Both gradients at 1x3x512^2 through the planar flow view every reference call site passes, against the oracle."""
    from sstem_restoration_b200 import SpatialTransformation, synth
    H = W = 512
    fl = (synth.random_fold_flow(H, W, 555)[0] if kind == "fold" else synth.noise_flow(H, W, 2.0, seed=7))[None]
    r = np.random.default_rng(512)
    mv = r.random((1, 3, H, W), dtype=np.float32)
    g = r.standard_normal((1, 3, H, W)).astype(np.float32)
    m = torch.from_numpy(mv).cuda().requires_grad_(True)
    base = torch.from_numpy(np.ascontiguousarray(fl.transpose(0, 3, 1, 2))).cuda().requires_grad_(True)
    SpatialTransformation(True)(m, base.permute(0, 2, 3, 1)).backward(torch.from_numpy(g).cuda())
    om, of = oracle.warp_torch_backward_restated(mv, fl, g)
    for got, want in ((m.grad, om), (base.grad.permute(0, 2, 3, 1), of)):
        assert np.abs(got.cpu().numpy() - want).max() <= 2e-5 * max(1.0, np.abs(want).max())


def test_spatial_transformation_backward_only_what_is_needed():
    from sstem_restoration_b200 import SpatialTransformation
    moving = torch.rand((1, 1, 8, 8), device="cuda", requires_grad=True)
    out = SpatialTransformation(True)(moving, torch.zeros((1, 8, 8, 2), device="cuda"))
    out.sum().backward()
    assert torch.equal(moving.grad, torch.ones_like(moving))       # identity flow: every pixel is its own (only) tap


# ---------------------------------------------------------------- numpy image_warp
@pytest.mark.parametrize("name", list(cases.image_warp_cases()))
def test_image_warp_matches_reference_bitwise(golden_dir, name):
    from sstem_restoration_b200 import image_warp
    ref = np.load(os.path.join(golden_dir, "warp_numpy_ref.npz"))[name]
    im, flow, mode = cases.image_warp_cases()[name]
    got = image_warp(im, flow, mode)
    assert got.dtype == np.uint8 and got.shape == ref.shape
    assert np.array_equal(got, ref), name
    got_t = image_warp(torch.from_numpy(im).cuda(), torch.from_numpy(flow).cuda(), mode)
    assert got_t.is_cuda and np.array_equal(got_t.cpu().numpy().reshape(ref.shape), ref)


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_image_warp_float_value_matches_oracle_bitwise(dtype, mode):
    from sstem_restoration_b200.warp import _image_warp_cuda
    r = np.random.default_rng(77)
    im = r.integers(0, 256, (2, 130, 257, 3)).astype(dtype)
    flow = (6.0 * r.standard_normal((2, 130, 257, 2))).astype(np.float32)
    u8, f = _image_warp_cuda(torch.from_numpy(im).cuda(), torch.from_numpy(flow).cuda(), mode, want_float=True)
    ref_u8, ref_f = oracle.image_warp_restated(im, flow, mode, return_float=True)
    assert np.array_equal(_bits(f.cpu().numpy()), _bits(ref_f.astype(np.float32)))
    assert np.array_equal(u8.cpu().numpy(), ref_u8)


def test_image_warp_errors_mirror_reference():
    from sstem_restoration_b200 import image_warp
    with pytest.raises(AttributeError):
        image_warp(np.zeros((1, 2, 2, 2, 2), np.uint8), np.zeros((2, 2, 2), np.float32))
    with pytest.raises(UnboundLocalError):
        image_warp(np.zeros((4, 4), np.uint8), np.zeros((4, 4, 2), np.float32), mode="cubic")
    with pytest.raises(TypeError):
        image_warp(np.zeros((4, 4), np.float64), np.zeros((4, 4, 2), np.float32))


def test_image_warp_simusff_config1_shape():
    """BASELINE config 1: uint8 256x256 EM-like section + gen_flow fold, bilinear."""
    from sstem_restoration_b200 import image_warp, synth
    sec = synth.em_section(256, 256, 0)
    flow, mask = synth.random_fold_flow(256, 256, 555)
    got = image_warp(sec, flow, "bilinear")
    assert np.array_equal(got, oracle.image_warp_restated(sec, flow, "bilinear"))


def test_image_warp_identity_at_full_size():
    from sstem_restoration_b200 import image_warp
    im = torch.randint(0, 256, (4096, 4096), dtype=torch.uint8, device="cuda")
    flow = torch.zeros((4096, 4096, 2), device="cuda")
    assert torch.equal(image_warp(im, flow), im)
    flow[..., 0] = 5.0
    got = image_warp(im, flow)
    assert torch.equal(got[:, :-5], im[:, 5:]) and torch.equal(got[:, -5:], im[:, -1:].expand(-1, 5))


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_image_warp_flow_slice_that_is_only_8_byte_aligned(dtype):
    """flows[i] of a [N,H,W,2] tensor with H*W odd starts 8 (not 16) bytes into a 16-byte line: the ABI's minimum flow
    alignment.  The kernel must not take its 16-byte flow loads there (it used to fault with 'misaligned address')."""
    from sstem_restoration_b200.warp import _image_warp_cuda
    r = np.random.default_rng(78)
    H, W = 33, 47                                         # H*W odd
    ims = r.integers(0, 256, (3, H, W, 3)).astype(dtype)
    flows = (4.0 * r.standard_normal((3, H, W, 2))).astype(np.float32)
    t_im, t_fl = torch.from_numpy(ims).cuda(), torch.from_numpy(flows).cuda()
    assert t_fl[1].data_ptr() % 16 == 8 and t_fl[1].is_contiguous()
    for i in range(3):
        u8, f = _image_warp_cuda(t_im[i], t_fl[i], "bilinear", want_float=True)
        ref_u8, ref_f = oracle.image_warp_restated(ims[i], flows[i], "bilinear", return_float=True)
        assert np.array_equal(u8.cpu().numpy(), ref_u8)
        assert np.array_equal(_bits(f.cpu().numpy()), _bits(ref_f.astype(np.float32)))
    torch.cuda.synchronize()
