"""Tap gradients of more than three channels on the persistent (third-generation) kernel.

The kernel handles three channels per launch; every later chunk adds its sum to grad_vertical / grad_horizontal in
place (one fp32 add per element).  So the gradients of a six-channel input must equal, bit for bit, the sum of the
gradients of its two three-channel halves, computed separately and added in the same order."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _tap_grads(x, v, h, g):
    import sstem_restoration_b200 as pkg
    v = v.clone().requires_grad_(True)
    h = h.clone().requires_grad_(True)
    pkg.SeparableConvolution.apply(x, v, h).backward(g)
    return v.grad, h.grad


@pytest.mark.parametrize("B,H,W", [(2, 512, 512), (1, 1001, 1004)])
def test_six_channels_accumulate_the_two_chunks_exactly(B, H, W):
    dev = "cuda"
    torch.manual_seed(21)
    x = torch.rand((B, 6, H + 50, W + 50), device=dev)
    v = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    h = torch.softmax(torch.randn((B, 51, H, W), device=dev), 1)
    g = torch.randn((B, 6, H, W), device=dev)
    gv, gh = _tap_grads(x, v, h, g)
    gv0, gh0 = _tap_grads(x[:, :3].contiguous(), v, h, g[:, :3].contiguous())
    gv1, gh1 = _tap_grads(x[:, 3:].contiguous(), v, h, g[:, 3:].contiguous())
    assert torch.equal(gv, gv0 + gv1)
    assert torch.equal(gh, gh0 + gh1)
