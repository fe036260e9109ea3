"""Adaptive separable local convolution: the reference's operator interface over
the sm_100a C ABI.

Mirrors, name for name and argument for argument,
  * ``SeparableConvolution`` (torch.autograd.Function) --
    libs/sepconv/SeparableConvolution.py:11-78 of the reference, and
  * ``FunctionSepconv`` / ``ModuleSepconv`` -- sff_scripts_interp/model/sepconv.py:152-164,
so ``IFNet`` (sff_scripts_interp/model/model_interp.py:47,94; sp_scripts_train/networks.py:70,120-123)
can bind ``self.separable_conv = SeparableConvolution.apply`` unchanged.

Behaviour kept: the shape / tap-count / contiguity ``assert``s
(SeparableConvolution.py:29-35), ``NotImplementedError`` for CPU tensors (:47-48),
a freshly allocated output on the input's device, a 3-tuple from backward.
Behaviour fixed (documented in include/sstem_b200.h): the backward channel sum
covers all C (the reference hard-codes 3), grad w.r.t. input is really computed
when requested (the reference returns zeros), ``needs_input_grad`` is honoured,
outputs are not redundantly zero-filled.
"""
from __future__ import annotations

import os

import torch

from . import _lib

_STRICT = os.environ.get("SSTEM_SEPCONV_STRICT", "0") not in ("", "0")


def set_strict_order(enabled: bool) -> None:
    """Evaluate the forward in the reference's exact fp32 summation order
    (bit-equal to kernel.cu:45-49; verification mode, slower)."""
    global _STRICT
    _STRICT = bool(enabled)


_GRAY = os.environ.get("SSTEM_SEPCONV_GRAY", "auto")       # off | assert | detect | auto
_AUTO_MIN_PIXELS = 1 << 19                                  # auto: detect from B*H*W of this size on (detection costs ~15 us + two empty launches)


def set_gray_replicated(mode) -> None:
    """Shortcut for the reference's actual inputs: grayscale sections replicated x3
    (sff_scripts_interp/data/data_provider.py:136-137), i.e. identical channel planes.

    ``"assert"``: the caller guarantees it.  ``"detect"``: every forward compares the planes ON THE DEVICE (one streaming
    kernel writing a device flag) and launches both the one-plane and the general path gated on that flag -- no host
    synchronisation; the backward reads the same flag.  ``"auto"`` (default): ``"detect"`` for calls of at least 2^19
    output pixels (where the detection's ~20 us are below 3 %), the general path below.  ``"off"``: always the general
    path.  Forward results are bit-identical either way; tap gradients agree to fp32 rounding."""
    global _GRAY
    mode = {True: "assert", False: "off", None: "off"}.get(mode, mode)
    if mode not in ("off", "assert", "detect", "auto"):
        raise ValueError("mode must be 'off', 'assert', 'detect' or 'auto'")
    _GRAY = mode


def _gray_mode(input, K) -> str:
    """-> 'off' | 'assert' | 'detect' for this call."""
    if _GRAY == "off" or _STRICT or input.size(1) < 2 or K != 51:
        return "off"
    if _GRAY == "auto":
        B, _, ih, iw = input.shape
        return "detect" if B * (ih - 50) * (iw - 50) >= _AUTO_MIN_PIXELS else "off"
    return _GRAY


def _is_gray(input) -> bool:
    """Host-side decision (used by the fused tail and the tiled forward): assert -> True; detect/auto -> compare (syncs)."""
    if _GRAY == "off" or _STRICT or input.size(1) < 2:
        return False
    if _GRAY == "assert":
        return True
    if _GRAY == "auto":
        return False
    return all(bool(torch.equal(input[:, 0], input[:, c])) for c in range(1, input.size(1)))


def _flags(gray: bool = False) -> int:
    f = _lib.SEPCONV_STRICT_ORDER if _STRICT else _lib.SEPCONV_DEFAULT
    return f | (_lib.SEPCONV_GRAY_REPLICATED if gray else 0)


def _stream_ptr(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _check_shapes(input, vertical, horizontal, filter_size=None):
    intInputHeight = input.size(2)
    intInputWidth = input.size(3)
    intFilterSize = min(vertical.size(1), horizontal.size(1))
    intOutputHeight = min(vertical.size(2), horizontal.size(2))
    intOutputWidth = min(vertical.size(3), horizontal.size(3))
    want = intFilterSize if filter_size is None else filter_size
    assert (intInputHeight - want == intOutputHeight - 1)
    assert (intInputWidth - want == intOutputWidth - 1)
    if filter_size is not None:
        assert (intFilterSize == filter_size)
    assert (input.is_contiguous() == True)
    assert (vertical.is_contiguous() == True)
    assert (horizontal.is_contiguous() == True)
    return intFilterSize, intOutputHeight, intOutputWidth


def _check_grad_output(grad_output, shape, like):
    """The kernels read the upstream gradient as contiguous float32 on the op's device: anything else
    (AMP half gradients, a double gradient handed to .backward(), another device) is converted or refused
    here instead of being misread."""
    if tuple(grad_output.shape) != tuple(shape):
        raise ValueError(f"sepconv backward: grad_output has shape {tuple(grad_output.shape)}, expected {tuple(shape)}")
    if grad_output.device != like.device:
        raise ValueError(f"sepconv backward: grad_output is on {grad_output.device}, the op ran on {like.device}")
    if grad_output.dtype != torch.float32:
        if not grad_output.dtype.is_floating_point:
            raise TypeError(f"sepconv backward: grad_output dtype {grad_output.dtype} is not a floating type")
        grad_output = grad_output.to(torch.float32)
    return grad_output.contiguous()


def _forward_impl(ctx, input, vertical, horizontal, filter_size):
    K, oh, ow = _check_shapes(input, vertical, horizontal, filter_size)
    if input.is_cuda == False:
        raise NotImplementedError()  # as the reference: CPU version not implemented
    if not (vertical.is_cuda and horizontal.is_cuda):
        raise NotImplementedError()
    if input.dtype != torch.float32 or vertical.dtype != torch.float32 or horizontal.dtype != torch.float32:
        raise TypeError("sepconv: float32 tensors required (the reference op is THCudaTensor = float)")
    assert vertical.shape == horizontal.shape, "vertical and horizontal must have the same shape"
    assert vertical.size(0) == input.size(0), "batch mismatch"
    B, C = input.size(0), input.size(1)
    output = torch.empty((B, C, oh, ow), dtype=input.dtype, device=input.device)
    ctx.gray = False
    ctx.gray_flag = None
    if output.numel() == 0:
        return output
    mode = _gray_mode(input, K)
    # the library launches on the device that owns `output`; only the stream has to be the caller's
    if mode == "detect":
        ctx.gray_flag = torch.empty(1, dtype=torch.int32, device=input.device)      # written and consumed on the device
        code = _lib.load().sstem_sepconv_forward_detect(
            input.data_ptr(), vertical.data_ptr(), horizontal.data_ptr(), output.data_ptr(),
            B, C, oh, ow, K, _flags(False), ctx.gray_flag.data_ptr(), _stream_ptr(input))
        if code:
            _lib.check(code, "sstem_sepconv_forward_detect")
        return output
    ctx.gray = mode == "assert"
    code = _lib.load().sstem_sepconv_forward(
        input.data_ptr(), vertical.data_ptr(), horizontal.data_ptr(), output.data_ptr(),
        B, C, oh, ow, K, _flags(ctx.gray), _stream_ptr(input))
    if code:
        _lib.check(code, "sstem_sepconv_forward")
    return output


def _backward_impl(ctx, grad_output):
    input, vertical, horizontal = ctx.saved_tensors
    need_in, need_v, need_h = ctx.needs_input_grad[:3]
    B, C = input.size(0), input.size(1)
    K, oh, ow = vertical.size(1), vertical.size(2), vertical.size(3)
    if grad_output.is_cuda == False:
        raise NotImplementedError()
    grad_output = _check_grad_output(grad_output, (B, C, oh, ow), input)
    grad_input = torch.empty_like(input) if need_in else None
    grad_vertical = torch.empty_like(vertical) if need_v else None
    grad_horizontal = torch.empty_like(horizontal) if need_h else None
    if (need_in or need_v or need_h) and grad_output.numel() > 0:
        flag = getattr(ctx, "gray_flag", None)
        ptrs = (grad_output.data_ptr(), input.data_ptr(), vertical.data_ptr(), horizontal.data_ptr(),
                grad_input.data_ptr() if need_in else None,
                grad_vertical.data_ptr() if need_v else None,
                grad_horizontal.data_ptr() if need_h else None)
        if flag is not None:
            code = _lib.load().sstem_sepconv_backward_detect(*ptrs, B, C, oh, ow, K, _flags(False), flag.data_ptr(), _stream_ptr(input))
        else:
            code = _lib.load().sstem_sepconv_backward(*ptrs, B, C, oh, ow, K, _flags(getattr(ctx, "gray", False)), _stream_ptr(input))
        if code:
            _lib.check(code, "sstem_sepconv_backward")
    return grad_input, grad_vertical, grad_horizontal


class SeparableConvolution(torch.autograd.Function):
    """Drop-in for libs/sepconv/SeparableConvolution.py:11-78 (51 taps, asserted)."""

    @staticmethod
    def forward(context, input, vertical, horizontal):
        context.save_for_backward(input, vertical, horizontal)
        return _forward_impl(context, input, vertical, horizontal, 51)

    @staticmethod
    def backward(context, grad_output):
        return _backward_impl(context, grad_output)


class _FunctionSepconv(torch.autograd.Function):
    """Drop-in for sff_scripts_interp/model/sepconv.py:76-150: tap count taken from
    the tensors (:83), and -- unlike the reference, whose backward raises
    NotImplementedError (:140-146) -- differentiable."""

    @staticmethod
    def forward(self, input, vertical, horizontal):
        self.save_for_backward(input, vertical, horizontal)
        return _forward_impl(self, input, vertical, horizontal, None)

    @staticmethod
    def backward(self, gradOutput):
        return _backward_impl(self, gradOutput)


def FunctionSepconv(tenInput, tenVertical, tenHorizontal):
    return _FunctionSepconv.apply(tenInput, tenVertical, tenHorizontal)


class ModuleSepconv(torch.nn.Module):
    def __init__(self):
        super(ModuleSepconv, self).__init__()

    def forward(self, tenInput, tenVertical, tenHorizontal):
        return _FunctionSepconv.apply(tenInput, tenVertical, tenHorizontal)


# ---------------------------------------------------------------------------------------------
# Fused interpolation tail (SURVEY.md section 8f, N1)
# ---------------------------------------------------------------------------------------------
def _frame_view(t):
    """A frame as the C ABI wants it: planes contiguous, any batch stride (x[:, :3] of a
    [B,6,H,W] tensor qualifies as is -- model_interp.py:56-57)."""
    B, C, H, W = t.shape
    ok = t.stride(3) == 1 and t.stride(2) == W and (C == 1 or t.stride(1) == H * W) and (B == 1 or t.stride(0) >= C * H * W)
    if not ok:
        t = t.contiguous()
    return t, (t.stride(0) if B > 1 else C * H * W)


class _InterpolationTail(torch.autograd.Function):
    @staticmethod
    def forward(ctx, i1, i2, k1v, k1h, k2v, k2h):
        for t in (i1, i2, k1v, k1h, k2v, k2h):
            if t.is_cuda == False:
                raise NotImplementedError()  # as SeparableConvolution.py:47-48: no CPU version
            if t.dtype != torch.float32:
                raise TypeError("interpolation_tail: float32 tensors required")
        assert i1.shape == i2.shape and i1.dim() == 4
        B, C, H, W = i1.shape
        for k in (k1v, k1h, k2v, k2h):
            assert tuple(k.shape) == (B, 51, H, W)          # SeparableConvolution.py:31 -- 51 taps
            assert (k.is_contiguous() == True)
        i1, bs1 = _frame_view(i1)
        i2, bs2 = _frame_view(i2)
        if bs1 != bs2:
            i1, i2 = i1.contiguous(), i2.contiguous()
            bs1 = bs2 = C * H * W
        # "detect" compares on the host here (the tail's general-channel mode already folds the channel mean into the window
        # load, so the shortcut is worth 20 %, not 2x); "auto" does not pay a synchronisation for that
        gray = C > 1 and (_GRAY == "assert" or (
            _GRAY == "detect" and all(bool(torch.equal(f[:, 0], f[:, c])) for f in (i1, i2) for c in range(1, C))))
        out = torch.empty((B, 1, H, W), dtype=torch.float32, device=i1.device)
        ctx.save_for_backward(i1, i2, k1v, k1h, k2v, k2h)
        ctx.tail = (bs1, gray)
        if out.numel() == 0:
            return out
        code = _lib.load().sstem_interp_tail_forward(
            i1.data_ptr(), i2.data_ptr(), bs1, k1v.data_ptr(), k1h.data_ptr(), k2v.data_ptr(), k2h.data_ptr(),
            out.data_ptr(), B, C, H, W, 51, _lib.SEPCONV_GRAY_REPLICATED if gray else 0, _stream_ptr(i1))
        if code:
            _lib.check(code, "sstem_interp_tail_forward")
        return out

    @staticmethod
    def backward(ctx, grad_output):
        i1, i2, k1v, k1h, k2v, k2h = ctx.saved_tensors
        bs, gray = ctx.tail
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            raise NotImplementedError("interpolation_tail: the frames are data; no gradient w.r.t. them "
                                      "(use SeparableConvolution on the padded frames for that)")
        need = ctx.needs_input_grad[2:6]
        B, C, H, W = i1.shape
        if grad_output.is_cuda == False:
            raise NotImplementedError()
        grad_output = _check_grad_output(grad_output, (B, 1, H, W), i1)
        grads = [torch.empty_like(k) if n else None for k, n in zip((k1v, k1h, k2v, k2h), need)]
        if any(need) and grad_output.numel() > 0:
            code = _lib.load().sstem_interp_tail_backward(
                grad_output.data_ptr(), i1.data_ptr(), i2.data_ptr(), bs,
                k1v.data_ptr(), k1h.data_ptr(), k2v.data_ptr(), k2h.data_ptr(),
                *[g.data_ptr() if g is not None else None for g in grads],
                B, C, H, W, 51, _lib.SEPCONV_GRAY_REPLICATED if gray else 0, _stream_ptr(i1))
            if code:
                _lib.check(code, "sstem_interp_tail_backward")
        return (None, None, *grads)


def interpolation_tail(i1, i2, k1v, k1h, k2v, k2h):
    """One launch for the expression every IFNet ends with (model_interp.py:90-97,
    sp_scripts_train/networks.py:116-123)::

        y = separable_conv(pad(i2), k2v, k2h) + separable_conv(pad(i1), k1v, k1h)   # pad = ReplicationPad2d(25)
        output = torch.mean(y, dim=1, keepdim=True)

    ``i1`` / ``i2``: UNPADDED frames [B,C,H,W] (views ``x[:, :3]`` / ``x[:, 3:6]`` are taken as they
    are); taps [B,51,H,W]; returns [B,1,H,W].  Differentiable w.r.t. the four tap tensors.  The
    gray x3 shortcut follows :func:`set_gray_replicated`.  Agrees with the unfused expression to
    fp32 rounding (the channel mean is taken before the convolution, which is linear in the image).
    """
    return _InterpolationTail.apply(i1, i2, k1v, k1h, k2v, k2h)


class ModuleInterpolationTail(torch.nn.Module):
    """``nn.Module`` form of :func:`interpolation_tail` (stateless)."""

    def forward(self, i1, i2, k1v, k1h, k2v, k2h):
        return _InterpolationTail.apply(i1, i2, k1v, k1h, k2v, k2h)


# ---------------------------------------------------------------------------------------------
# Tile-major taps (SURVEY.md section 8f, N2)
# ---------------------------------------------------------------------------------------------
def taps_to_tiled(taps: torch.Tensor) -> torch.Tensor:
    """[B,51,H,W] taps -> the tile-major layout ``[B, ceil(H/8), ceil(W/8), 51, 8, 8]`` (zeros outside the image) that
    :func:`sepconv_forward_tiled` consumes: all 51 taps of an 8x8 pixel tile are 13 KB of contiguous memory.  This is
    the layout a tap producer -- the last ``Conv2d(51,51,3)`` of ``IFNet._kernel_module``,
    sff_scripts_interp/model/model_interp.py:129-137 -- should write; the conversion exists for producers that cannot
    (and for the parity tests)."""
    if taps.is_cuda == False:
        raise NotImplementedError()
    if taps.dtype != torch.float32 or taps.dim() != 4 or taps.size(1) != 51:
        raise TypeError("taps_to_tiled: float32 [B,51,H,W] required")
    taps = taps.contiguous()
    B, _, H, W = taps.shape
    out = torch.empty((B, (H + 7) // 8, (W + 7) // 8, 51, 8, 8), dtype=torch.float32, device=taps.device)
    if out.numel():
        code = _lib.load().sstem_taps_to_tiled(taps.data_ptr(), out.data_ptr(), B, H, W, _stream_ptr(taps))
        if code:
            _lib.check(code, "sstem_taps_to_tiled")
    return out


def taps_from_tiled(tiled: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """Inverse of :func:`taps_to_tiled`: tile-major ``[B, ceil(H/8), ceil(W/8), 51, 8, 8]`` -> [B,51,H,W] (the entries
    outside the image are not read)."""
    if tiled.is_cuda == False:
        raise NotImplementedError()
    want = ((H + 7) // 8, (W + 7) // 8, 51, 8, 8)
    if tiled.dtype != torch.float32 or tiled.dim() != 6 or tuple(tiled.shape[1:]) != want:
        raise TypeError(f"taps_from_tiled: float32 [B,{','.join(map(str, want))}] required for H={H}, W={W}")
    tiled = tiled.contiguous()
    B = tiled.size(0)
    out = torch.empty((B, 51, H, W), dtype=torch.float32, device=tiled.device)
    if out.numel():
        code = _lib.load().sstem_taps_from_tiled(tiled.data_ptr(), out.data_ptr(), B, H, W, _stream_ptr(tiled))
        if code:
            _lib.check(code, "sstem_taps_from_tiled")
    return out


def _check_tiled(what, input, vertical_tiled, horizontal_tiled):
    for t in (input, vertical_tiled, horizontal_tiled):
        if t.is_cuda == False:
            raise NotImplementedError()
        if t.dtype != torch.float32:
            raise TypeError(f"{what}: float32 tensors required")
    assert (input.is_contiguous() == True) and (vertical_tiled.is_contiguous() == True) and (horizontal_tiled.is_contiguous() == True)
    B, C, IH, IW = input.shape
    H, W = IH - 50, IW - 50
    want = (B, (H + 7) // 8, (W + 7) // 8, 51, 8, 8)
    assert tuple(vertical_tiled.shape) == want and tuple(horizontal_tiled.shape) == want, f"tiled taps must be {want}"
    return B, C, H, W


def _forward_tiled(input, vertical_tiled, horizontal_tiled, out, accumulate, gray):
    B, C, H, W = out.shape
    if out.numel():
        flags = (_lib.SEPCONV_GRAY_REPLICATED if gray else 0) | (_lib.SEPCONV_ACCUMULATE if accumulate else 0)
        code = _lib.load().sstem_sepconv_forward_tiled(input.data_ptr(), vertical_tiled.data_ptr(), horizontal_tiled.data_ptr(),
                                                       out.data_ptr(), B, C, H, W, 51, flags, _stream_ptr(input))
        if code:
            _lib.check(code, "sstem_sepconv_forward_tiled")
    return out


def _backward_tiled(grad_output, input, vertical_tiled, horizontal_tiled, need_in, need_v, need_h, gray):
    """-> (grad_input, grad_vertical_tiled, grad_horizontal_tiled), None where not needed."""
    B, C, IH, IW = input.shape
    grad_output = _check_grad_output(grad_output, (B, C, IH - 50, IW - 50), input)
    grad_input = torch.empty_like(input) if need_in else None
    grad_v = torch.empty_like(vertical_tiled) if need_v else None
    grad_h = torch.empty_like(horizontal_tiled) if need_h else None
    if (need_in or need_v or need_h) and grad_output.numel() > 0:
        code = _lib.load().sstem_sepconv_backward_tiled(
            grad_output.data_ptr(), input.data_ptr(), vertical_tiled.data_ptr(), horizontal_tiled.data_ptr(),
            grad_input.data_ptr() if need_in else None, grad_v.data_ptr() if need_v else None,
            grad_h.data_ptr() if need_h else None, B, C, IH - 50, IW - 50, 51,
            _lib.SEPCONV_GRAY_REPLICATED if gray else 0, _stream_ptr(input))
        if code:
            _lib.check(code, "sstem_sepconv_backward_tiled")
    return grad_input, grad_v, grad_h


def sepconv_forward_tiled(input: torch.Tensor, vertical_tiled: torch.Tensor, horizontal_tiled: torch.Tensor, out=None,
                          accumulate: bool = False) -> torch.Tensor:
    """``SeparableConvolution.apply(input, vertical, horizontal)`` with both tap tensors in the tile-major layout of
    :func:`taps_to_tiled`; forward only (no autograd graph: use :class:`SeparableConvolutionTiled` for gradients);
    bit-identical to the [B,51,H,W] path.  Follows :func:`set_gray_replicated`.
    ``out`` / ``accumulate``: write into (add to) an existing [B,C,H,W] tensor -- the second frame of the interpolation
    tail (the general path only: the gray shortcut writes its replicas from one register)."""
    B, C, H, W = _check_tiled("sepconv_forward_tiled", input, vertical_tiled, horizontal_tiled)
    if out is None:
        if accumulate:
            raise ValueError("sepconv_forward_tiled: accumulate needs an existing `out`")
        out = torch.empty((B, C, H, W), dtype=torch.float32, device=input.device)
    else:
        assert tuple(out.shape) == (B, C, H, W) and out.dtype == torch.float32 and (out.is_contiguous() == True) and out.device == input.device
    gray = out.numel() > 0 and (not accumulate) and _is_gray(input)
    return _forward_tiled(input, vertical_tiled, horizontal_tiled, out, accumulate, gray)


class SeparableConvolutionTiled(torch.autograd.Function):
    """:class:`SeparableConvolution` with both tap tensors in the tile-major layout of :func:`taps_to_tiled`:
    ``SeparableConvolutionTiled.apply(input, vertical_tiled, horizontal_tiled)`` -> [B,C,H,W].  The tap gradients come
    out tile-major as well (zero outside the image); with taps that run the same kernel on the [B,51,H,W] path they are
    bit-identical to :class:`SeparableConvolution`'s.  The gray x3 shortcut is decided once, on the host, in the forward
    (:func:`set_gray_replicated`; ``"auto"`` does not pay a synchronisation for it) and reused by the backward."""

    @staticmethod
    def forward(ctx, input, vertical_tiled, horizontal_tiled):
        B, C, H, W = _check_tiled("SeparableConvolutionTiled", input, vertical_tiled, horizontal_tiled)
        out = torch.empty((B, C, H, W), dtype=torch.float32, device=input.device)
        ctx.gray = out.numel() > 0 and _is_gray(input)
        ctx.save_for_backward(input, vertical_tiled, horizontal_tiled)
        return _forward_tiled(input, vertical_tiled, horizontal_tiled, out, False, ctx.gray)

    @staticmethod
    def backward(ctx, grad_output):
        input, vertical_tiled, horizontal_tiled = ctx.saved_tensors
        if grad_output.is_cuda == False:
            raise NotImplementedError()
        return _backward_tiled(grad_output, input, vertical_tiled, horizontal_tiled, *ctx.needs_input_grad[:3], ctx.gray)


def frame_mean_pad(frame: torch.Tensor, pad: int = 25, gray=None) -> torch.Tensor:
    """``ReplicationPad2d(pad)(frame.mean(1, keepdim=True))`` in one launch: the one-plane frame the tile-major
    interpolation tail convolves.  ``frame`` [B,C,H,W] (a channel slice ``x[:, :3]`` of the network input is taken as it
    is); ``gray`` (default: :func:`set_gray_replicated` mode ``"assert"``): the planes are identical copies, plane 0 is used."""
    if frame.is_cuda == False:
        raise NotImplementedError()
    if frame.dtype != torch.float32 or frame.dim() != 4:
        raise TypeError("frame_mean_pad: float32 [B,C,H,W] required")
    frame, bs = _frame_view(frame)
    B, C, H, W = frame.shape
    if gray is None:
        gray = C > 1 and _GRAY == "assert"
    out = torch.empty((B, 1, H + 2 * pad, W + 2 * pad), dtype=torch.float32, device=frame.device)
    if out.numel():
        code = _lib.load().sstem_frame_mean_pad(frame.data_ptr(), bs, out.data_ptr(), B, C, H, W, pad,
                                                _lib.SEPCONV_GRAY_REPLICATED if gray else 0, _stream_ptr(frame))
        if code:
            _lib.check(code, "sstem_frame_mean_pad")
    return out


def interpolation_tail_tiled(i1, i2, k1v_tiled, k1h_tiled, k2v_tiled, k2h_tiled) -> torch.Tensor:
    """:func:`interpolation_tail` for tap tensors in the tile-major layout (what :class:`ModuleTapProducer` emits): the whole
    tail of ``IFNet.forward`` (model_interp.py:90-97) without a [B,51,H,W] tensor anywhere.  Forward only (no autograd
    graph: :class:`ModuleInterpolationTailTiled` is the differentiable form).

    mean_c sepconv(pad(i_c)) = sepconv(pad(mean_c i_c)), so each frame is reduced to one replicate-padded plane
    (:func:`frame_mean_pad`) and convolved by the persistent one-channel kernel; the second frame accumulates into the first
    frame's output.  Returns [B,1,H,W]; agrees with :func:`interpolation_tail` to fp32 rounding."""
    p2, p1 = frame_mean_pad(i2), frame_mean_pad(i1)
    out = sepconv_forward_tiled(p2, k2v_tiled, k2h_tiled)
    return sepconv_forward_tiled(p1, k1v_tiled, k1h_tiled, out=out, accumulate=True)


class _InterpolationTailTiled(torch.autograd.Function):
    @staticmethod
    def forward(ctx, i1, i2, k1v, k1h, k2v, k2h):
        p2, p1 = frame_mean_pad(i2), frame_mean_pad(i1)
        out = sepconv_forward_tiled(p2, k2v, k2h)
        ctx.save_for_backward(p1, p2, k1v, k1h, k2v, k2h)
        return sepconv_forward_tiled(p1, k1v, k1h, out=out, accumulate=True)

    @staticmethod
    def backward(ctx, grad_output):
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            raise NotImplementedError("interpolation_tail_tiled: the frames are data; no gradient w.r.t. them "
                                      "(use SeparableConvolutionTiled on the padded frames for that)")
        if grad_output.is_cuda == False:
            raise NotImplementedError()
        p1, p2, k1v, k1h, k2v, k2h = ctx.saved_tensors
        n1v, n1h, n2v, n2h = ctx.needs_input_grad[2:6]
        # out = sepconv(p2, k2) + sepconv(p1, k1) on the one-plane mean frames: each frame's taps see grad_output as is
        _, g2v, g2h = _backward_tiled(grad_output, p2, k2v, k2h, False, n2v, n2h, False)
        _, g1v, g1h = _backward_tiled(grad_output, p1, k1v, k1h, False, n1v, n1h, False)
        return None, None, g1v, g1h, g2v, g2h


class ModuleInterpolationTailTiled(torch.nn.Module):
    """Differentiable :func:`interpolation_tail_tiled` (stateless): the same forward, and the four tap gradients in the
    tile-major layout, two one-plane tiled backward calls on the padded mean frames.  The frames get no gradient
    (``NotImplementedError`` if one is asked for, as :func:`interpolation_tail`)."""

    def forward(self, i1, i2, k1v_tiled, k1h_tiled, k2v_tiled, k2h_tiled):
        return _InterpolationTailTiled.apply(i1, i2, k1v_tiled, k1h_tiled, k2v_tiled, k2h_tiled)
