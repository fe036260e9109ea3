"""Tap producer: the last two layers of the reference's ``IFNet._kernel_module``

    nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) -> nn.Conv2d(51, 51, 3, 1, 1)

(sff_scripts_interp/model/model_interp.py:18, 130-137; four instances, :34-37, run at :86-89) as one sm_100a kernel
(csrc/tapconv.cu: tcgen05 TF32 implicit GEMM, the upsample folded into the operand producer), writing the taps in the
layout of ``Conv2d`` or directly tile-major for :func:`sstem_restoration_b200.sepconv_forward_tiled`.
:func:`tap_conv3x3` is forward only (the stack-restoration path, c5); :class:`TapConv3x3Function` and
``ModuleTapProducer(trainable=True)`` add the backward (tcgen05 kernels as well) for training.

The three half-resolution ``Conv2d -> ReLU`` layers in front of them run on :func:`branch_conv3x3` (csrc/tapconv.cu, the same
tcgen05 machinery fed by TMA from a chunk-major activation layout), their gradients on :func:`branch_conv3x3_backward`;
:class:`ModuleTapBranch` is the whole branch, forward only by default and trainable with ``trainable=True``.  No CPU /
PyTorch fallback.
"""
import torch

from . import _lib


def _stream_ptr(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _pack(weight: torch.Tensor, name: str, entry: str, elems: str, max_cin: int, max_cout: int, tag=True) -> torch.Tensor:
    """``weight`` packed by the C entry point ``entry`` into an image of ``elems()`` floats, for the public function ``name``
    and within its channel limits.  ``tag``: the image carries (cin, cout) as ``_sstem_cin_cout``."""
    if weight.is_cuda == False:
        raise NotImplementedError()
    if weight.dtype != torch.float32 or weight.dim() != 4 or tuple(weight.shape[2:]) != (3, 3):
        raise TypeError(f"{name}: float32 [cout, cin, 3, 3] required")
    cout, cin = weight.shape[:2]
    if cin > max_cin or cout > max_cout:
        raise ValueError(f"{name}: cin <= {max_cin} and cout <= {max_cout} required")
    lib = _lib.load()
    packed = torch.empty(getattr(lib, elems)(), dtype=torch.float32, device=weight.device)
    code = getattr(lib, entry)(weight.contiguous().data_ptr(), packed.data_ptr(), cin, cout, _stream_ptr(weight))
    if code:
        _lib.check(code, entry)
    if tag:
        packed._sstem_cin_cout = (int(cin), int(cout))
    return packed


def pack_tap_conv_weight(weight: torch.Tensor) -> torch.Tensor:
    """``Conv2d.weight`` ``[cout<=64, cin<=52, 3, 3]`` -> the kernel's resident image (118 KB, TF32-rounded).  Pack once per
    layer, reuse for every call."""
    return _pack(weight, "pack_tap_conv_weight", "sstem_tap_conv3x3_pack_weights", "sstem_tap_conv3x3_packed_elems", 52, 64)


def pack_tap_conv_weight_adjoint(weight: torch.Tensor) -> torch.Tensor:
    """``Conv2d.weight`` ``[cout<=52, cin<=52, 3, 3]`` -> the resident image of the adjoint convolution's weight
    ``W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]`` (cout -> cin channels), which the input gradient runs."""
    # untagged: tap_conv3x3 would read the weight's (cin, cout), not the adjoint's (cout, cin)
    return _pack(weight, "pack_tap_conv_weight_adjoint", "sstem_tap_conv3x3_pack_weights_adjoint", "sstem_tap_conv3x3_packed_elems",
                 52, 52, tag=False)


def tap_conv3x3(x: torch.Tensor, packed_weight: torch.Tensor, bias=None, cin=None, cout=None, upsample=True, tiled=False) -> torch.Tensor:
    """``conv2d(upsample2x(x), weight, bias, stride 1, padding 1)`` (``upsample=False``: the convolution alone).

    x ``[B, cin, h, w]`` float32 contiguous; ``packed_weight`` from :func:`pack_tap_conv_weight`.  Returns ``[B, cout, H, W]``
    or, with ``tiled=True`` (cout == 51), the tile-major taps ``[B, ceil(H/8), ceil(W/8), 51, 8, 8]``."""
    if x.is_cuda == False:
        raise NotImplementedError()
    if x.dtype != torch.float32 or x.dim() != 4:
        raise TypeError("tap_conv3x3: float32 [B, cin, h, w] required")
    assert x.is_contiguous() == True
    if torch.is_grad_enabled() and x.requires_grad:
        # forward only: returning a tensor without a graph would silently cut the gradient of everything upstream
        raise NotImplementedError("tap_conv3x3 is forward only (the stack-restoration path): call it under torch.no_grad() or detach its input")
    if cin is None or cout is None:
        cin, cout = getattr(packed_weight, "_sstem_cin_cout", (None, None))
        if cin is None:
            raise ValueError("tap_conv3x3: pass cin / cout (the packed weight does not carry them)")
    B, c, h, w = x.shape
    if c != cin:
        raise ValueError(f"tap_conv3x3: x has {c} channels, the weight {cin}")
    H, W = (2 * h, 2 * w) if upsample else (h, w)
    if tiled:
        if cout != 51:
            raise ValueError("tap_conv3x3: the tile-major layout is defined for 51 taps")
        out = torch.empty((B, (H + 7) // 8, (W + 7) // 8, 51, 8, 8), dtype=torch.float32, device=x.device)
    else:
        out = torch.empty((B, cout, H, W), dtype=torch.float32, device=x.device)
    if out.numel():
        flags = (_lib.TAPCONV_UPSAMPLE2X if upsample else 0) | (_lib.TAPCONV_TILED if tiled else 0)
        code = _lib.load().sstem_tap_conv3x3(x.data_ptr(), packed_weight.data_ptr(), bias.contiguous().data_ptr() if bias is not None else None,
                                             out.data_ptr(), B, cin, cout, h, w, flags, _stream_ptr(x))
        if code:
            _lib.check(code, "sstem_tap_conv3x3")
    return out


class TapConv3x3Function(torch.autograd.Function):
    """``conv2d(upsample2x(x), weight, bias, padding 1)`` with its backward, over the raw ``Conv2d`` ``weight`` ``[cout, cin, 3,
    3]`` (cin, cout <= 52) and ``bias`` (or None):

        TapConv3x3Function.apply(x, weight, bias, upsample=True, tiled=False, packed=None, packed_adjoint=None)

    ``tiled=True`` (cout == 51) returns the tile-major taps of :func:`tap_conv3x3`, and the backward then takes their
    gradient tile-major, as :class:`SeparableConvolutionTiled` / :class:`ModuleInterpolationTailTiled` return it.
    ``packed`` / ``packed_adjoint``: images of ``weight`` from :func:`pack_tap_conv_weight` /
    :func:`pack_tap_conv_weight_adjoint`, packed here when not given.  The gradients are TF32 (the reference layer's
    precision under torch's default ``allow_tf32``), deterministic; inputs that need none get ``None``."""

    @staticmethod
    def forward(ctx, x, weight, bias=None, upsample=True, tiled=False, packed=None, packed_adjoint=None):
        if packed is None:
            packed = pack_tap_conv_weight(weight.detach())
        if packed_adjoint is None and ctx.needs_input_grad[0]:
            packed_adjoint = pack_tap_conv_weight_adjoint(weight.detach())
        cout, cin = weight.shape[:2]
        y = tap_conv3x3(x, packed, None if bias is None else bias.detach(), cin=cin, cout=cout, upsample=upsample, tiled=tiled)
        ctx.save_for_backward(x)
        ctx.packed_adjoint, ctx.upsample, ctx.tiled, ctx.cin_cout, ctx.has_bias = packed_adjoint, upsample, tiled, (cin, cout), bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        cin, cout = ctx.cin_cout
        need_x, need_w, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        gx = torch.empty_like(x) if need_x else None
        gw = torch.empty((cout, cin, 3, 3), dtype=torch.float32, device=x.device) if need_w else None
        gb = torch.empty(cout, dtype=torch.float32, device=x.device) if need_b else None
        if (need_x or need_w or need_b) and x.numel():
            gy = gy.contiguous()
            B, _, h, w = x.shape
            flags = (_lib.TAPCONV_UPSAMPLE2X if ctx.upsample else 0) | (_lib.TAPCONV_TILED if ctx.tiled else 0)
            ptr = lambda t: None if t is None else t.data_ptr()
            code = _lib.load().sstem_tap_conv3x3_backward(gy.data_ptr(), x.data_ptr(), ptr(ctx.packed_adjoint) if need_x else None,
                                                          ptr(gx), ptr(gw), ptr(gb), B, cin, cout, h, w, flags, _stream_ptr(x))
            if code:
                _lib.check(code, "sstem_tap_conv3x3_backward")
        return gx, gw, gb, None, None, None, None


class ModuleTapProducer(torch.nn.Module):
    """Drop-in for the tail ``nn.Sequential(upsample, Conv2d(51, 51, 3, 1, 1))`` of ``_kernel_module``: holds ``weight`` /
    ``bias`` under the names of ``nn.Conv2d`` (so the reference layer's state_dict loads), packs the weight on first use
    and whenever it changes.  Forward only by default (an input that requires grad raises); ``trainable=True`` runs
    :class:`TapConv3x3Function`, so gradients reach ``x``, ``weight`` and ``bias``."""

    def __init__(self, in_channels=51, out_channels=51, upsample=True, tiled=False, trainable=False):
        super().__init__()
        self.weight = torch.nn.Parameter(torch.empty(out_channels, in_channels, 3, 3))
        self.bias = torch.nn.Parameter(torch.zeros(out_channels))
        torch.nn.init.kaiming_uniform_(self.weight, a=5 ** 0.5)
        self.upsample, self.tiled, self.trainable = upsample, tiled, trainable
        self._packed = self._packed_adjoint = None
        self._versions = {}

    def _cached(self, name, pack, device):
        """``self.<name>``, packed again from the weight whenever the weight or the device changed."""
        key = (self.weight._version, self.weight.data_ptr())
        packed = getattr(self, name)
        if packed is None or self._versions.get(name) != key or packed.device != device:
            setattr(self, name, pack(self.weight.detach()))
            self._versions[name] = key
        return getattr(self, name)

    def forward(self, x):
        packed = self._cached("_packed", pack_tap_conv_weight, x.device)
        if not self.trainable:
            return tap_conv3x3(x, packed, self.bias.detach(), upsample=self.upsample, tiled=self.tiled)
        need_adjoint = torch.is_grad_enabled() and x.requires_grad
        adjoint = self._cached("_packed_adjoint", pack_tap_conv_weight_adjoint, x.device) if need_adjoint else None
        return TapConv3x3Function.apply(x, self.weight, self.bias, self.upsample, self.tiled, packed, adjoint)


def pack_branch_conv_weight(weight: torch.Tensor) -> torch.Tensor:
    """``Conv2d.weight`` ``[cout<=64, cin<=64, 3, 3]`` -> the resident image of :func:`branch_conv3x3` (144 KB,
    TF32-rounded).  Pack once per layer, reuse for every call."""
    return _pack(weight, "pack_branch_conv_weight", "sstem_branch_conv3x3_pack_weights", "sstem_branch_conv3x3_packed_elems", 64, 64)


def pack_branch_conv_weight_adjoint(weight: torch.Tensor) -> torch.Tensor:
    """``Conv2d.weight`` ``[cout<=64, cin<=64, 3, 3]`` -> the resident image of the adjoint convolution's weight
    ``W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]`` (cout -> cin channels), which the input gradient of
    :func:`branch_conv3x3_backward` runs.  It carries (cin, cout) of ``weight``."""
    return _pack(weight, "pack_branch_conv_weight_adjoint", "sstem_branch_conv3x3_pack_weights_adjoint",
                 "sstem_branch_conv3x3_packed_elems", 64, 64)


def _layout_shape(B, c, h, w, chunked):
    """The shape of ``c`` channels: chunk-major ``[B, C8/4, h, w, 4]`` (C8 = c rounded up to 8), else ``[B, c, h, w]``."""
    return (B, (c + 7) // 8 * 2, h, w, 4) if chunked else (B, c, h, w)


def branch_conv3x3(x: torch.Tensor, packed: torch.Tensor, bias=None, relu=True, chunked_in=False, chunked_out=False) -> torch.Tensor:
    """``relu?(conv2d(x, weight, bias, stride 1, padding 1))``, one half-resolution layer of a tap branch.

    ``packed`` comes from :func:`pack_branch_conv_weight` (it carries cin / cout).  x is ``[B, cin, h, w]`` or, with
    ``chunked_in``, chunk-major ``[B, C8/4, h, w, 4]`` (C8 = cin rounded up to 8; values TF32-rounded, padding channels 0:
    what ``chunked_out`` returns).  Returns ``[B, cout, h, w]`` in full fp32 or, with ``chunked_out``, chunk-major.
    Forward only."""
    if x.is_cuda == False:
        raise NotImplementedError()
    if x.dtype != torch.float32 or x.dim() != (5 if chunked_in else 4) or not x.is_contiguous():
        raise TypeError("branch_conv3x3: contiguous float32 [B, cin, h, w] (chunk-major: [B, C8/4, h, w, 4]) required")
    if torch.is_grad_enabled() and x.requires_grad:
        raise NotImplementedError("branch_conv3x3 is forward only: call it under torch.no_grad() or detach its input")
    cin, cout = getattr(packed, "_sstem_cin_cout", (None, None))
    if cin is None:
        raise ValueError("branch_conv3x3: the packed weight must come from pack_branch_conv_weight")
    B, c, h, w = x.shape[:4]
    if tuple(x.shape) != _layout_shape(B, cin, h, w, chunked_in):
        raise ValueError(f"branch_conv3x3: x {tuple(x.shape)} does not match the weight's {cin} input channels")
    out = torch.empty(_layout_shape(B, cout, h, w, chunked_out), dtype=torch.float32, device=x.device)
    if out.numel():
        flags = ((_lib.BRANCH_RELU if relu else 0) | (_lib.BRANCH_IN_CHUNKED if chunked_in else 0)
                 | (_lib.BRANCH_OUT_CHUNKED if chunked_out else 0))
        code = _lib.load().sstem_branch_conv3x3(x.data_ptr(), packed.data_ptr(), bias.contiguous().data_ptr() if bias is not None else None,
                                                out.data_ptr(), B, cin, cout, h, w, flags, _stream_ptr(x))
        if code:
            _lib.check(code, "sstem_branch_conv3x3")
    return out


def branch_conv3x3_backward(grad_out, y, x, packed_adjoint, cin, cout, relu=True, chunked_in=False, chunked_out=False,
                            need=(True, True, True)):
    """Gradients of ``y = relu?(conv2d(x, weight, bias, stride 1, padding 1))`` (:func:`branch_conv3x3`) from ``grad_out``
    ``[B, cout, h, w]``: returns ``(grad_x [B, cin, h, w], grad_weight [cout, cin, 3, 3], grad_bias [cout])``, ``None``
    for each one ``need`` does not ask for.

    ``y`` and ``x`` are the forward's output and input in the layouts it wrote and read (``chunked_out`` / ``chunked_in``:
    chunk-major ``[B, C8/4, h, w, 4]``); ``y`` is only read with ``relu`` (zero gradient where ``y <= 0``, as torch's ReLU backward)
    and may then be None otherwise.  ``packed_adjoint`` from :func:`pack_branch_conv_weight_adjoint` (None when grad_x is
    not needed).  TF32 products, fp32 sums, deterministic; grad_bias sums the unrounded masked gradient."""
    if grad_out.is_cuda == False or x.is_cuda == False:
        raise NotImplementedError()
    if grad_out.dtype != torch.float32 or x.dtype != torch.float32:
        raise TypeError("branch_conv3x3_backward: float32 tensors required")
    B, _, h, w = x.shape[:4]
    if tuple(grad_out.shape) != (B, cout, h, w):
        raise ValueError(f"branch_conv3x3_backward: grad_out {tuple(grad_out.shape)} is not [{B}, {cout}, {h}, {w}]")
    if tuple(x.shape) != _layout_shape(B, cin, h, w, chunked_in) or not x.is_contiguous():
        raise ValueError(f"branch_conv3x3_backward: x {tuple(x.shape)} does not match cin = {cin} (chunked_in={chunked_in})")
    if relu and (y is None or tuple(y.shape) != _layout_shape(B, cout, h, w, chunked_out) or not y.is_contiguous()):
        raise ValueError("branch_conv3x3_backward: relu needs the forward's contiguous output y in its layout")
    need_x, need_w, need_b = need
    if need_x and (packed_adjoint is None or getattr(packed_adjoint, "_sstem_cin_cout", None) != (cin, cout)):
        raise ValueError("branch_conv3x3_backward: grad_x needs packed_adjoint = pack_branch_conv_weight_adjoint(weight)")
    gx = torch.empty((B, cin, h, w), dtype=torch.float32, device=x.device) if need_x else None
    gw = torch.empty((cout, cin, 3, 3), dtype=torch.float32, device=x.device) if need_w else None
    gb = torch.empty(cout, dtype=torch.float32, device=x.device) if need_b else None
    if (need_x or need_w or need_b) and grad_out.numel():
        grad_out = grad_out.contiguous()
        flags = ((_lib.BRANCH_RELU if relu else 0) | (_lib.BRANCH_IN_CHUNKED if chunked_in else 0)
                 | (_lib.BRANCH_OUT_CHUNKED if chunked_out else 0))
        ptr = lambda t: None if t is None else t.data_ptr()
        code = _lib.load().sstem_branch_conv3x3_backward(grad_out.data_ptr(), ptr(y) if relu else None, x.data_ptr(),
                                                         ptr(packed_adjoint) if need_x else None, ptr(gx), ptr(gw), ptr(gb),
                                                         B, cin, cout, h, w, flags, _stream_ptr(x))
        if code:
            _lib.check(code, "sstem_branch_conv3x3_backward")
    return gx, gw, gb


def _branch_convs(x, packs, biases):
    """The three half-resolution ``Conv2d -> ReLU`` layers of a tap branch, chained on :func:`branch_conv3x3`: NCHW x ->
    chunk-major -> chunk-major -> NCHW.  Returns the output of each layer."""
    a1 = branch_conv3x3(x, packs[0], biases[0], relu=True, chunked_in=False, chunked_out=True)
    a2 = branch_conv3x3(a1, packs[1], biases[1], relu=True, chunked_in=True, chunked_out=True)
    a3 = branch_conv3x3(a2, packs[2], biases[2], relu=True, chunked_in=True, chunked_out=False)
    return a1, a2, a3


class _TapBranchConvs(torch.autograd.Function):
    """:func:`_branch_convs` with its backward: the forward keeps x, the two chunk-major activations and the output; the
    backward runs :func:`branch_conv3x3_backward` once per layer, last layer first."""

    @staticmethod
    def forward(ctx, x, w0, b0, w2, b2, w4, b4, packs, adjoints):
        a1, a2, a3 = _branch_convs(x, packs, (b0.detach(), b2.detach(), b4.detach()))
        ctx.save_for_backward(x, a1, a2, a3)
        ctx.adjoints, ctx.shapes = adjoints, tuple(tuple(t.shape[:2]) for t in (w0, w2, w4))
        return a3

    @staticmethod
    def backward(ctx, g3):
        x, a1, a2, a3 = ctx.saved_tensors
        need = ctx.needs_input_grad
        (c1, c0), (c2, _), (c3, _) = ctx.shapes
        adj = ctx.adjoints
        g2, gw4, gb4 = branch_conv3x3_backward(g3, a3, a2, adj[2], c2, c3, chunked_in=True, chunked_out=False,
                                               need=(True, need[5], need[6]))
        g1, gw2, gb2 = branch_conv3x3_backward(g2, a2, a1, adj[1], c1, c2, chunked_in=True, chunked_out=True,
                                               need=(True, need[3], need[4]))
        gx, gw0, gb0 = branch_conv3x3_backward(g1, a1, x, adj[0] if need[0] else None, c0, c1, chunked_in=False, chunked_out=True,
                                               need=(need[0], need[1], need[2]))
        return gx, gw0, gb0, gw2, gb2, gw4, gb4, None, None


class _BranchConv(ModuleTapProducer):
    """The parameters of one ``Conv2d(cin, cout, 3, 1, 1) -> ReLU`` of a tap branch, with the cache of their packed images
    (:meth:`ModuleTapProducer._cached`); :class:`ModuleTapBranch` runs the three layers together."""

    def __init__(self, in_channels, out_channels):
        super().__init__(in_channels, out_channels, upsample=False)


class ModuleTapBranch(torch.nn.Module):
    """Drop-in for a whole tap branch, ``IFNet._kernel_module`` (model_interp.py:129-137):

        Conv2d(in, mid, 3, 1, 1), ReLU, Conv2d(mid, mid, 3, 1, 1), ReLU, Conv2d(mid, taps, 3, 1, 1), ReLU,
        Upsample(scale_factor=2, mode='bilinear', align_corners=True), Conv2d(taps, taps, 3, 1, 1)

    Its state_dict has the keys of that ``nn.Sequential`` (``0.*``, ``2.*``, ``4.*``, ``7.*``), so
    ``m.load_state_dict(net.upconv51_1.state_dict())`` loads a reference branch.  The three half-resolution layers run on
    :func:`branch_conv3x3` (NCHW in, chunk-major between them, ``[B, taps, h, w]`` out), the last two on the tap producer;
    ``tiled=True`` returns the taps tile-major (:func:`sstem_restoration_b200.sepconv_forward_tiled`'s layout).  Forward
    only by default: an input that requires grad raises.  ``trainable=True`` runs the three layers with their backward
    (:func:`branch_conv3x3_backward`) and the producer as ``ModuleTapProducer(trainable=True)``: gradients reach all
    eight parameters, and ``x`` when it requires grad."""

    def __init__(self, in_channels=64, mid_channels=64, taps=51, tiled=True, trainable=False):
        super().__init__()
        self.in_channels, self.trainable = in_channels, trainable
        self.add_module("0", _BranchConv(in_channels, mid_channels))
        self.add_module("2", _BranchConv(mid_channels, mid_channels))
        self.add_module("4", _BranchConv(mid_channels, taps))
        self.add_module("7", ModuleTapProducer(taps, taps, upsample=True, tiled=tiled, trainable=trainable))

    def forward(self, x):
        if not self.trainable and torch.is_grad_enabled() and x.requires_grad:
            raise NotImplementedError("ModuleTapBranch is forward only: call it under torch.no_grad() or detach its input")
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise ValueError(f"ModuleTapBranch: x [B, {self.in_channels}, h, w] required, got {tuple(x.shape)}")
        convs = [getattr(self, k) for k in ("0", "2", "4")]
        packs = tuple(c._cached("_packed", pack_branch_conv_weight, x.device) for c in convs)
        if self.trainable:
            adjoints = (tuple(c._cached("_packed_adjoint", pack_branch_conv_weight_adjoint, x.device) for c in convs)
                        if torch.is_grad_enabled() else None)
            a = _TapBranchConvs.apply(x.contiguous(), *(t for c in convs for t in (c.weight, c.bias)), packs, adjoints)
        else:
            a = _branch_convs(x.contiguous(), packs, tuple(c.bias.detach() for c in convs))[2]
        return getattr(self, "7")(a)
