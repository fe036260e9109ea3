"""Element-wise parity at BASELINE's real sizes against the REFERENCE'S OWN CUDA
(libs/sepconv/src/SeparableConvolution_kernel.cu:25-52,77-150), not only against size-independent properties.

  c2   in[1,3,306,306],   v,h[1,51,256,256]    (whole section; KPN-like raw taps, |out| ~ 1e1..1e2)
  c3   in[2,3,562,562],   v,h[2,51,512,512]    (two samples of the training batch)
  c4   in[1,3,2098,2098], v,h[1,51,2048,2048]

tests/golden/sepconv_fullsize_ref.npz holds SHA-256 digests of these inputs and of the reference kernel's forward,
grad_vertical and grad_horizontal on them (tests/golden/make_fullsize_parity_golden.py).  Whole tensors that match those
digests bit for bit ARE the reference's outputs: the forward is the STRICT_ORDER forward of this package, the tap
gradients are the CPU oracle's reference-order restatement (oracle/sepconv_oracle.c).  Against them, for each case, the
default (re-associated) forward / grad_vertical / grad_horizontal satisfy protocol P1 or P2 of SURVEY.md 8(c) element-wise
over the whole tensor (|new - ref| <= 1e-5 * max(1, max|ref|) and err(new, fp64) <= max(1.25 * err(ref, fp64), 2e-6 * scale));
grad_input (absent in the reference) is compared with the fp64 adjoint.  fp64 truths are evaluated on the GPU with
plain torch shifts (2 601 slice-multiply-adds); at c2 the CPU oracle's forward is checked against the same reference
output, which ties the three together.  Dense-tap accumulation across every tile seam of the full grid is what these
cases add over the <= 64x64 oracle cases.

The measured max-abs figures are written to gpurun_out/parity_fullsize.json (copied to profiles/ when run by hand).
"""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu

TOL = 1e-5
K = 51
_REPORT = {}


def _record(name, **kw):
    _REPORT.setdefault(name, {}).update({k: float(v) for k, v in kw.items()})
    try:
        out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "parity_fullsize.json"), "w") as f:
            json.dump(_REPORT, f, indent=1, sort_keys=True)
    except OSError:
        pass


def _em_input(B, H, W, dev, seed):
    """gray x3, /255, ReplicationPad2d(25) -- what sff_scripts_interp/inference.py:71-77 + model_interp.py:46 feed."""
    from sstem_restoration_b200 import synth
    secs = [synth.em_section(min(H, 1024), min(W, 1024), seed + b) for b in range(B)]
    t = torch.from_numpy(np.stack(secs)).to(dev).float().div_(255.0)
    if H > 1024 or W > 1024:                              # tile the 1024^2 texture (generation cost), then perturb per pixel
        t = t.repeat(1, -(-H // 1024), -(-W // 1024))[:, :H, :W].contiguous()
        g = torch.Generator(device=dev).manual_seed(seed)
        t = (t + 0.02 * torch.randn(t.shape, device=dev, generator=g)).clamp_(0, 1)
    t = torch.nn.functional.pad(t[:, None], (25, 25, 25, 25), mode="replicate")
    return t.expand(B, 3, H + 50, W + 50).contiguous()


def _kpn_like_taps(B, H, W, dev, seed, vmax):
    """Raw taps with the structure of IFNet._kernel_module's tail (model_interp.py:129-137: ... -> Upsample x2 ->
    Conv2d(51,51,3)): half-resolution features, bilinear upsampling, a random 3x3 51->51 conv, no normalisation; scaled to
    the magnitudes the reference's random-init KPN shows on this input (|v| <= 3.7, |h| <= 7.4 -- SURVEY 0.5)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    f = torch.randn((B, K, H // 2, W // 2), device=dev, generator=g)
    f = torch.nn.functional.avg_pool2d(f, 5, stride=1, padding=2)
    f = torch.nn.functional.interpolate(f, size=(H, W), mode="bilinear", align_corners=False)
    w = torch.randn((K, K, 3, 3), device=dev, generator=g) / (3.0 * K ** 0.5)
    t = torch.nn.functional.conv2d(f, w, padding=1)
    t = t + 0.05 * torch.randn(t.shape, device=dev, generator=g)
    return (t * (vmax / t.abs().max())).contiguous()


def _unit_taps(B, H, W, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.softmax(torch.randn((B, K, H, W), device=dev, generator=g), 1).contiguous()


def case_inputs(name, dev):
    """(input, vertical, horizontal, grad_output) of one entry of CASES."""
    B, H, W, kind = CASES[name]
    inp = _em_input(B, H, W, dev, seed=700 + H)
    if kind == "kpn":
        v, h = _kpn_like_taps(B, H, W, dev, 31, 3.7), _kpn_like_taps(B, H, W, dev, 32, 7.4)
    else:
        v, h = _unit_taps(B, H, W, dev, 33), _unit_taps(B, H, W, dev, 34)
    g = torch.randn((B, 3, H, W), device=dev, generator=torch.Generator(device=dev).manual_seed(99))
    return inp, v, h, g


def tail_inputs(dev):
    """Two gray x3 512^2 frames and four unit-tap tensors: the reference's actual call."""
    B, H, W = 1, 512, 512
    return _em_input(B, H, W, dev, seed=41), _em_input(B, H, W, dev, seed=43), [_unit_taps(B, H, W, dev, 50 + i) for i in range(4)]


def sha256(*tensors):
    """SHA-256 of the tensors' bytes, in order, as uint8[32] (the format of the digests in the golden fixtures)."""
    d = hashlib.sha256()
    for t in tensors:
        d.update(t.detach().contiguous().cpu().numpy())
    return np.frombuffer(d.digest(), np.uint8)


def _check_digest(key, what, *tensors):
    want = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sepconv_fullsize_ref.npz"))[key + "_sha256"]
    assert np.array_equal(sha256(*tensors), want), f"{key}: {what}"


def _strict_forward(inp, v, h):
    import sstem_restoration_b200 as pkg
    pkg.set_strict_order(True)
    try:
        return pkg.SeparableConvolution.apply(inp, v, h)
    finally:
        pkg.set_strict_order(False)


def _truth_f64(inp, v, h, g):
    """fp64 forward, grad_v, grad_h, grad_input by shifted slices (2 601 steps), all on the GPU."""
    B, C, IH, IW = inp.shape
    H, W = IH - K + 1, IW - K + 1
    i64, v64, h64, g64 = inp.double(), v.double(), h.double(), g.double()
    out = torch.zeros((B, C, H, W), dtype=torch.float64, device=inp.device)
    gv = torch.zeros((B, K, H, W), dtype=torch.float64, device=inp.device)
    gh = torch.zeros_like(gv)
    gi = torch.zeros_like(i64)
    for fy in range(K):
        r = torch.zeros_like(out)
        gvf = torch.zeros((B, H, W), dtype=torch.float64, device=inp.device)
        gw = g64 * v64[:, fy:fy + 1]                       # g * v[fy]
        for fx in range(K):
            win = i64[:, :, fy:fy + H, fx:fx + W]
            r.addcmul_(win, h64[:, fx:fx + 1])
            t = (g64 * win).sum(1)                         # t[fy][fx] = sum_c g_c * in_c
            gvf.addcmul_(t, h64[:, fx])
            gh[:, fx].addcmul_(t, v64[:, fy])
            gi[:, :, fy:fy + H, fx:fx + W].addcmul_(gw, h64[:, fx:fx + 1])
        out.addcmul_(r, v64[:, fy:fy + 1])
        gv[:, fy] = gvf
    return out, gv, gh, gi


def _p_check(name, what, got, ref32, ref64):
    scale = max(1.0, float(ref64.abs().max()))
    err_vs_ref = float((got.double() - ref32.double()).abs().max())
    err_new = float((got.double() - ref64).abs().max())
    err_ref = float((ref32.double() - ref64).abs().max())
    _record(name, **{what + "_max_abs_vs_ref": err_vs_ref, what + "_err_new_f64": err_new, what + "_err_ref_f64": err_ref,
                     what + "_scale": scale})
    assert err_vs_ref <= TOL * scale, f"{name} {what}: |new-ref|={err_vs_ref:.3e} scale={scale:.3g}"
    assert err_new <= max(1.25 * err_ref, 2e-6 * scale), f"{name} {what}: err(new,f64)={err_new:.3e} > err(ref,f64)={err_ref:.3e}"


CASES = {
    # name: (B, H, W, taps kind)
    "c2_256_kpnlike": (1, 256, 256, "kpn"),
    "c2_256_unit": (1, 256, 256, "unit"),
    "c3_2x512_unit": (2, 512, 512, "unit"),
    "c3_1x512_kpnlike": (1, 512, 512, "kpn"),
    "c4_2048_unit": (1, 2048, 2048, "unit"),
}


@pytest.mark.parametrize("name", list(CASES))
def test_fullsize_forward_and_tap_gradients_vs_reference_cuda(name):
    import sstem_restoration_b200 as pkg
    B, H, W, kind = CASES[name]
    dev = torch.device("cuda")
    inp, v, h, g = case_inputs(name, dev)
    _check_digest(name + "_inputs", "not the inputs the stored reference outputs were computed from", inp, v, h, g)

    # strict order: bit-equal to the reference kernel over the whole tensor
    ref_out = _strict_forward(inp, v, h)
    _check_digest(name + "_out", "strict-order forward is not bit-equal to the reference kernel", ref_out)
    # the reference kernel's tap gradients: the oracle's reference-order restatement, bit-equal over the whole tensor
    ni, nv, nh, ng = (t.cpu().numpy() for t in (inp, v, h, g))
    ref_gv = torch.from_numpy(oracle.sepconv_grad_vertical_reforder(ng, ni, nh)).to(dev)
    _check_digest(name + "_gv", "oracle grad_vertical is not bit-equal to the reference kernel", ref_gv)
    ref_gh = torch.from_numpy(oracle.sepconv_grad_horizontal_reforder(ng, ni, nv)).to(dev)
    _check_digest(name + "_gh", "oracle grad_horizontal is not bit-equal to the reference kernel", ref_gh)

    # default kernels
    iv = inp.clone().requires_grad_(True)
    vv, hh = v.clone().requires_grad_(True), h.clone().requires_grad_(True)
    out = pkg.SeparableConvolution.apply(iv, vv, hh)
    out.backward(g)
    t_out, t_gv, t_gh, t_gi = _truth_f64(inp, v, h, g)
    _p_check(name, "fwd", out.detach(), ref_out, t_out)
    _p_check(name, "gv", vv.grad, ref_gv, t_gv)
    _p_check(name, "gh", hh.grad, ref_gh, t_gh)
    gscale = max(1.0, float(t_gi.abs().max()))
    gi_err = float((iv.grad.double() - t_gi).abs().max())
    _record(name, gi_err_f64=gi_err, gi_scale=gscale)
    assert gi_err <= TOL * gscale, f"{name} gi: {gi_err:.3e} (scale {gscale:.3g})"

    if H <= 256:                                          # tie the CPU oracle's forward to the same reference output (seconds in C)
        assert np.array_equal(oracle.sepconv_forward_reforder(ni, nv, nh).view(np.uint32), ref_out.cpu().numpy().view(np.uint32))
    del t_out, t_gv, t_gh, t_gi, ref_gv, ref_gh
    torch.cuda.empty_cache()


def test_fullsize_gray_shortcut_and_fused_tail_vs_reference_cuda():
    """The reference's actual call (gray x3 frames): shortcut forward bit-identical to the general path at 512^2, and the
    fused tail within 1e-5 of mean_c(ref(i2) + ref(i1)) computed by the reference kernel."""
    import sstem_restoration_b200 as pkg
    dev = torch.device("cuda")
    inp, inp2, taps = tail_inputs(dev)
    _check_digest("tail_512_inputs", "not the inputs the stored reference outputs were computed from", inp, inp2, *taps)
    ref1 = _strict_forward(inp, taps[0], taps[1])
    _check_digest("tail_512_ref1", "strict-order forward is not bit-equal to the reference kernel", ref1)
    ref2 = _strict_forward(inp2, taps[2], taps[3])
    _check_digest("tail_512_ref2", "strict-order forward is not bit-equal to the reference kernel", ref2)
    general = pkg.SeparableConvolution.apply(inp, taps[0], taps[1])
    pkg.set_gray_replicated("assert")
    try:
        gray = pkg.SeparableConvolution.apply(inp, taps[0], taps[1])
    finally:
        pkg.set_gray_replicated("off")
    assert torch.equal(gray, general)
    assert float((general - ref1).abs().max()) <= TOL
    f1, f2 = inp[:, :, 25:-25, 25:-25].contiguous(), inp2[:, :, 25:-25, 25:-25].contiguous()
    fused = pkg.interpolation_tail(f1, f2, taps[0], taps[1], taps[2], taps[3])
    expect = torch.mean(ref2 + ref1, dim=1, keepdim=True)
    err = float((fused - expect).abs().max())
    _record("tail_512", fused_vs_reference_expression=err)
    assert err <= TOL
