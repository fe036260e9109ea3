"""CPU: argument checks of the tiled tap-gradient entry points (sstem_sepconv_backward_tiled, sstem_taps_from_tiled) run
before any CUDA call, so they need no GPU."""
import ctypes

import pytest
import torch


@pytest.fixture()
def lib(built_lib):
    from sstem_restoration_b200 import _lib
    return _lib.load()


def test_backward_tiled_argument_errors(lib):
    buf = ctypes.create_string_buffer(256)
    p = (ctypes.addressof(buf) + 15) & ~15                 # 16-byte aligned host address: never dereferenced
    bwd = lib.sstem_sepconv_backward_tiled
    assert bwd(p, p, p, p, p, p, p, 1, 3, 8, 8, 51, 0, None) == -4                   # valid arguments: host memory refused
    assert bwd(None, p, p, p, p, p, p, 1, 3, 8, 8, 51, 0, None) == -1                # grad_output NULL
    assert bwd(p, None, p, p, p, p, p, 1, 3, 8, 8, 51, 0, None) == -1                # input NULL
    assert bwd(p, p, None, p, p, p, p, 1, 3, 8, 8, 51, 0, None) == -1                # vertical taps NULL
    assert bwd(p, p, p, None, p, p, p, 1, 3, 8, 8, 51, 0, None) == -1                # horizontal taps NULL
    assert bwd(p, p, p, p, None, None, None, 1, 3, 8, 8, 51, 0, None) == -1          # nothing to compute
    assert bwd(p, p, p, p, None, p, None, 0, 3, 8, 8, 51, 0, None) == -2             # B = 0
    assert bwd(p, p, p, p, None, p, None, 1, 0, 8, 8, 51, 0, None) == -2             # C = 0
    assert bwd(p, p, p, p, None, p, None, 1, 3, -1, 8, 51, 0, None) == -2            # H < 0
    assert bwd(p, p, p, p, None, p, None, 1, 3, 8, (1 << 24) + 1, 51, 0, None) == -2 # W out of range
    assert bwd(p, p, p, p, None, p, None, 1, 65536, 8, 8, 51, 0, None) == -2         # C out of range
    assert bwd(p, p, p, p, None, p, None, 1, 3, 8, 8, 49, 0, None) == -2             # the tiled layout has 51 taps
    assert bwd(p, p, p, p, None, p, None, 1, 3, 8, 8, 51, 1, None) == -5             # STRICT_ORDER: forward only
    assert bwd(p, p, p, p, None, p, None, 1, 3, 8, 8, 51, 4, None) == -5             # ACCUMULATE: forward only
    assert bwd(p, p, p, p, None, p, None, 1, 3, 8, 8, 51, 2, None) == -4             # GRAY_REPLICATED is accepted
    assert bwd(p + 2, p, p, p, None, p, None, 1, 3, 8, 8, 51, 0, None) == -3         # grad_output not 4-byte aligned
    assert bwd(p, p + 1, p, p, None, p, None, 1, 3, 8, 8, 51, 0, None) == -3         # input not 4-byte aligned
    assert bwd(p, p, p + 4, p, None, p, None, 1, 3, 8, 8, 51, 0, None) == -3         # tiled taps 16-byte aligned
    assert bwd(p, p, p, p + 8, None, p, None, 1, 3, 8, 8, 51, 0, None) == -3
    assert bwd(p, p, p, p, None, p + 4, None, 1, 3, 8, 8, 51, 0, None) == -3         # tiled gradients 16-byte aligned
    assert bwd(p, p, p, p, None, None, p + 4, 1, 3, 8, 8, 51, 0, None) == -3
    assert bwd(p, p, p, p, p + 2, None, None, 1, 3, 8, 8, 51, 0, None) == -3         # grad_input 4-byte aligned
    assert bwd(p, p, p, p, p + 4, None, None, 1, 3, 8, 8, 51, 0, None) == -4         # (and needs no more)


def test_taps_from_tiled_argument_errors(lib):
    buf = ctypes.create_string_buffer(256)
    p = (ctypes.addressof(buf) + 15) & ~15
    conv = lib.sstem_taps_from_tiled
    assert conv(p, p, 1, 8, 8, None) == -4
    assert conv(None, p, 1, 8, 8, None) == -1
    assert conv(p, None, 1, 8, 8, None) == -1
    assert conv(p, p, 0, 8, 8, None) == -2
    assert conv(p, p, 1, 0, 8, None) == -2
    assert conv(p, p, 1, 8, (1 << 24) + 1, None) == -2
    assert conv(p + 4, p, 1, 8, 8, None) == -3                                        # tiled source 16-byte aligned
    assert conv(p, p + 2, 1, 8, 8, None) == -3


def test_tiled_autograd_forms_refuse_cpu_tensors(built_lib):
    import sstem_restoration_b200 as pkg
    inp = torch.zeros((1, 3, 58, 58))
    tiled = torch.zeros((1, 1, 1, 51, 8, 8))
    with pytest.raises(NotImplementedError):               # as SeparableConvolution.py:47-48: no CPU version
        pkg.SeparableConvolutionTiled.apply(inp, tiled, tiled)
    with pytest.raises(NotImplementedError):
        pkg.ModuleInterpolationTailTiled()(torch.zeros((1, 3, 8, 8)), torch.zeros((1, 3, 8, 8)), *([tiled] * 4))
    with pytest.raises(NotImplementedError):
        pkg.taps_from_tiled(tiled, 8, 8)
