"""CPU: the tap branch backward's C ABI (argument checks, version), its Python entry points without a GPU, and the fp64
restatement the GPU tests compare against (tests/_tapconv_bwd_ref.py without the upsample, fed g = gy * (y > 0))."""
import ctypes

import numpy as np
import pytest
import torch

from tests import _tapconv_bwd_ref as ref


def test_abi_version_is_7(built_lib):
    from sstem_restoration_b200 import _lib
    assert _lib.ABI_VERSION == 7
    assert _lib.load().sstem_abi_version() == 7


def test_backward_argument_errors(built_lib):
    from sstem_restoration_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1024)
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16       # 16-byte aligned host memory
    relu, cin_ck, out_ck = _lib.BRANCH_RELU, _lib.BRANCH_IN_CHUNKED, _lib.BRANCH_OUT_CHUNKED
    pk = lib.sstem_branch_conv3x3_pack_weights_adjoint
    assert pk(None, p, 64, 64, None) == -1
    assert pk(p, None, 64, 64, None) == -1
    assert pk(p, p, 65, 64, None) == -2                                   # cin <= 64
    assert pk(p, p, 64, 65, None) == -2                                   # cout <= 64
    assert pk(p, p, 0, 64, None) == -2
    assert pk(p, p, 64, 0, None) == -2
    assert pk(p + 2, p, 64, 64, None) == -3
    assert pk(p, p + 4, 64, 64, None) == -3                               # packed image 16-byte aligned
    assert pk(p, p, 64, 64, None) == -4                                   # host memory
    bw = lib.sstem_branch_conv3x3_backward
    #        grad_out y  x  adj gx gw gb  B  cin cout h  w  flags
    assert bw(None, p, p, p, p, p, p, 1, 64, 64, 4, 4, relu, None) == -1
    assert bw(p, None, p, p, p, p, p, 1, 64, 64, 4, 4, relu, None) == -1          # RELU needs y
    assert bw(p, p, None, p, p, p, p, 1, 64, 64, 4, 4, relu, None) == -1
    assert bw(p, p, p, None, p, p, p, 1, 64, 64, 4, 4, relu, None) == -1          # grad_x needs the adjoint image
    assert bw(p, p, p, p, p, p, p, 1, 64, 64, 4, 4, 8, None) == -5                # unknown flag bit
    assert bw(p, p, p, p, p, p, p, 1, 65, 64, 4, 4, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 1, 64, 65, 4, 4, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 1, 0, 64, 4, 4, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 1, 64, 0, 4, 4, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 0, 64, 64, 4, 4, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 1, 64, 64, 0, 4, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 1, 64, 64, 4, -1, relu, None) == -2
    assert bw(p, p, p, p, p, p, p, 1, 64, 64, 1 << 23, 4, relu, None) == -2
    assert bw(p + 2, p, p, p, p, p, p, 1, 64, 64, 4, 4, relu, None) == -3
    assert bw(p, p + 2, p, p, p, p, p, 1, 64, 64, 4, 4, relu, None) == -3
    assert bw(p, p + 4, p, p, p, p, p, 1, 64, 64, 4, 4, relu | out_ck, None) == -3   # chunk-major y: 16 B
    assert bw(p, p, p + 4, p, p, p, p, 1, 64, 64, 4, 4, relu | cin_ck, None) == -3  # chunk-major x: 16 B
    assert bw(p, p, p, p + 4, p, p, p, 1, 64, 64, 4, 4, relu, None) == -3           # packed adjoint: 16 B
    assert bw(p, p, p, p, p + 1, p, p, 1, 64, 64, 4, 4, relu, None) == -3
    assert bw(p, p, p, p, p, p + 1, p, 1, 64, 64, 4, 4, relu, None) == -3
    assert bw(p, p, p, p, p, p, p + 1, 1, 64, 64, 4, 4, relu, None) == -3
    assert bw(p, p, p, p, p, p, p, 1, 64, 64, 4, 4, relu, None) == -4              # host memory
    assert bw(p, None, p, None, None, p, None, 1, 64, 64, 4, 4, 0, None) == -4     # no ReLU: y unused; grad_x not asked
    assert bw(p, p, p, None, None, None, None, 1, 64, 64, 4, 4, relu, None) == 0   # nothing asked: nothing done


def test_python_entry_points_refuse_cpu_tensors(built_lib):
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    import sstem_restoration_b200 as pkg
    with pytest.raises(NotImplementedError):
        pkg.pack_branch_conv_weight_adjoint(torch.zeros((64, 64, 3, 3)))
    x = torch.zeros((1, 64, 4, 4))
    with pytest.raises(NotImplementedError):
        pkg.branch_conv3x3_backward(torch.zeros((1, 64, 4, 4)), x, x, None, 64, 64)
    with pytest.raises(NotImplementedError):
        pkg.ModuleTapBranch(trainable=True)(x)
    with pytest.raises(NotImplementedError):
        pkg.ModuleTapBranch(trainable=True)(x.clone().requires_grad_(True))


def test_trainable_module_keeps_the_reference_state_dict_keys():
    import sstem_restoration_b200 as pkg
    nn = torch.nn
    ref_seq = nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 51, 3, 1, 1),
                            nn.ReLU(), nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True), nn.Conv2d(51, 51, 3, 1, 1))
    want = ref_seq.state_dict()
    m = pkg.ModuleTapBranch(trainable=True)
    assert list(m.state_dict()) == list(want)
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == {k: tuple(v.shape) for k, v in want.items()}
    m.load_state_dict(want)
    assert all(torch.equal(m.state_dict()[k], v) for k, v in want.items())
    assert getattr(m, "7").trainable and len(list(m.parameters())) == 8


@pytest.mark.parametrize("B,cin,cout,h,w", [(1, 5, 7, 6, 5), (2, 8, 3, 4, 9), (1, 3, 4, 1, 1), (2, 4, 6, 7, 1)])
def test_restated_layer_backward_matches_torch_cpu_autograd(B, cin, cout, h, w):
    r = np.random.default_rng(B * 100 + cin * 10 + cout + h + w)
    x = torch.from_numpy(r.standard_normal((B, cin, h, w))).requires_grad_(True)
    wt = torch.from_numpy(r.standard_normal((cout, cin, 3, 3))).requires_grad_(True)
    b = torch.from_numpy(r.standard_normal(cout)).requires_grad_(True)
    gy = torch.from_numpy(r.standard_normal((B, cout, h, w)))
    y = torch.relu(torch.nn.functional.conv2d(x, wt, b, padding=1))
    y.backward(gy)
    g = (gy * (y.detach() > 0)).numpy()
    gx, gw, gb = ref.tap_conv3x3_backward_restated(g, x.detach().numpy(), wt.detach().numpy(), upsample=False)
    for got, want in ((x.grad, gx), (wt.grad, gw), (b.grad, gb)):
        assert got.shape == want.shape
        assert np.abs(got.numpy() - want).max() <= 1e-12 * max(1.0, np.abs(want).max())
