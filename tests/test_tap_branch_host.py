"""CPU: the tap branch's C ABI (argument checks, sizes) and Python entry points, no GPU needed."""
import ctypes

import pytest
import torch


def test_branch_conv_argument_errors(built_lib):
    from sstem_restoration_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(256)
    p = (ctypes.addressof(buf) + 15) // 16 * 16
    relu, cin_ck, out_ck = _lib.BRANCH_RELU, _lib.BRANCH_IN_CHUNKED, _lib.BRANCH_OUT_CHUNKED
    assert lib.sstem_branch_conv3x3_pack_weights(None, p, 64, 64, None) == -1
    assert lib.sstem_branch_conv3x3_pack_weights(p, None, 64, 64, None) == -1
    assert lib.sstem_branch_conv3x3_pack_weights(p, p, 65, 64, None) == -2                 # cin <= 64
    assert lib.sstem_branch_conv3x3_pack_weights(p, p, 64, 65, None) == -2                 # cout <= 64
    assert lib.sstem_branch_conv3x3_pack_weights(p, p, 0, 64, None) == -2
    assert lib.sstem_branch_conv3x3_pack_weights(p + 2, p, 64, 64, None) == -3
    assert lib.sstem_branch_conv3x3_pack_weights(p, p + 4, 64, 64, None) == -3             # packed image 16-byte aligned
    assert lib.sstem_branch_conv3x3(None, p, None, p, 1, 64, 64, 4, 4, relu, None) == -1
    assert lib.sstem_branch_conv3x3(p, None, None, p, 1, 64, 64, 4, 4, relu, None) == -1
    assert lib.sstem_branch_conv3x3(p, p, None, None, 1, 64, 64, 4, 4, relu, None) == -1
    assert lib.sstem_branch_conv3x3(p, p, None, p, 1, 64, 64, 4, 4, 8, None) == -5           # unknown flag bit
    assert lib.sstem_branch_conv3x3(p, p, None, p, 1, 65, 64, 4, 4, relu, None) == -2
    assert lib.sstem_branch_conv3x3(p, p, None, p, 1, 64, 65, 4, 4, relu, None) == -2
    assert lib.sstem_branch_conv3x3(p, p, None, p, 0, 64, 64, 4, 4, relu, None) == -2
    assert lib.sstem_branch_conv3x3(p, p, None, p, 1, 64, 64, 0, 4, relu, None) == -2
    assert lib.sstem_branch_conv3x3(p, p, None, p, 1, 64, 64, 4, -1, relu, None) == -2
    assert lib.sstem_branch_conv3x3(p + 2, p, None, p, 1, 64, 64, 4, 4, relu, None) == -3
    assert lib.sstem_branch_conv3x3(p + 4, p, None, p, 1, 64, 64, 4, 4, relu | cin_ck, None) == -3   # chunk-major x: 16 B
    assert lib.sstem_branch_conv3x3(p, p + 4, None, p, 1, 64, 64, 4, 4, relu, None) == -3
    assert lib.sstem_branch_conv3x3(p, p, None, p + 4, 1, 64, 64, 4, 4, relu | out_ck, None) == -3   # chunk-major out: 16 B
    assert lib.sstem_branch_conv3x3(p, p, p + 2, p, 1, 64, 64, 4, 4, relu, None) == -3


def test_branch_conv_sizes(built_lib):
    from sstem_restoration_b200 import _lib
    lib = _lib.load()
    assert lib.sstem_branch_conv3x3_packed_elems() == 9 * 16 * 64 * 4
    for B, c, h, w in ((1, 64, 1024, 1024), (2, 17, 5, 7), (16, 51, 256, 256), (1, 1, 1, 1), (3, 8, 9, 2)):
        assert lib.sstem_chunked_elems(B, c, h, w) == B * ((c + 7) // 8 * 8) * h * w
    assert lib.sstem_chunked_elems(0, 64, 4, 4) == 0
    assert lib.sstem_chunked_elems(1, 64, 4, -4) == 0


def test_python_entry_points_refuse_cpu_tensors(built_lib):
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    import sstem_restoration_b200 as pkg
    with pytest.raises(NotImplementedError):
        pkg.pack_branch_conv_weight(torch.zeros((64, 64, 3, 3)))
    with pytest.raises(NotImplementedError):
        pkg.branch_conv3x3(torch.zeros((1, 64, 4, 4)), torch.zeros(36864))
    with pytest.raises(NotImplementedError):
        pkg.ModuleTapBranch()(torch.zeros((1, 64, 4, 4)))


def _reference_branch():
    nn = torch.nn
    return nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 51, 3, 1, 1),
                         nn.ReLU(), nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True), nn.Conv2d(51, 51, 3, 1, 1))


def test_module_state_dict_matches_the_reference_branch():
    import sstem_restoration_b200 as pkg
    ref = _reference_branch().state_dict()
    got = pkg.ModuleTapBranch().state_dict()
    assert list(got) == list(ref)
    assert {k: tuple(v.shape) for k, v in got.items()} == {k: tuple(v.shape) for k, v in ref.items()}
    m = pkg.ModuleTapBranch()
    m.load_state_dict(ref)
    assert all(torch.equal(m.state_dict()[k], v) for k, v in ref.items())
