"""The TMA flow warp (``warp_torch_tma_kernel``, csrc/warp.cu) against the oracle, bit for bit, in every window tier.

Every reference call site of ``SpatialTransformation`` passes a planar flow view (``pred_flow.permute(0,2,3,1)``), and that
layout runs the TMA kernel; its ``STITCH`` instantiation is ``warp_and_stitch``, the config-5 stack job.  Each 8x64 output
tile of that kernel takes one of five code paths, chosen from the bounding box of its taps: the small (12x72), mid
(16x80) or large (24x96) shared-memory window, the out-of-line partial tile (a 24x96 window centred on the mean tap,
in or out decided per pixel; not in ``STITCH``), or plain global gathers.  ``_tiers`` restates that choice in numpy so
that each flow below is known to reach the path it is meant for (the CPU test pins the counts), and the GPU tests hold
every path to ``oracle.warp_torch_restated`` / ``oracle.warp_stitch_restated``.
"""
import functools

import numpy as np
import pytest
import torch

import oracle
from sstem_restoration_b200 import synth

# Tile and window geometry of warp_torch_tma_kernel (csrc/warp.cu: WT_TH x WT_TW, WT_SH x WT_SW, WT_MH x WT_MW,
# WT_BH x WT_BW, and the `moderate` bound (WT_BW + 32) x (2 * WT_BH) of the partial tier).  Test-only: a change of the
# kernel's geometry changes these in the same commit.
TILE_H, TILE_W = 8, 64
WINDOWS = ((12, 72), (16, 80), (24, 96), (48, 128))         # (rows, columns): small, mid, large, partial
TIERS = ("small", "mid", "large", "partial", "gather")


def _tiers(flow):
    """flow [H,W,2] float32 -> [tiles_y, tiles_x] tier index into TIERS, as warp_torch_tma_kernel chooses it."""
    H, W, _ = flow.shape
    one = np.float32(1)
    x = (flow[..., 0] + np.arange(W, dtype=np.float32)[None]) + one           # torch_tap, float32 op order
    y = (flow[..., 1] + np.arange(H, dtype=np.float32)[:, None]) + one
    xf, yf = np.floor(x), np.floor(y)
    # the float clamp to the 1-px zero-padded image, then image coordinates of the first and last tap (-1 .. W / H)
    xa = np.clip(xf, 0, W + 1).astype(np.int64) - 1
    xb = np.clip(xf + 1, 0, W + 1).astype(np.int64) - 1
    ya = np.clip(yf, 0, H + 1).astype(np.int64) - 1
    yb = np.clip(yf + 1, 0, H + 1).astype(np.int64) - 1
    th, tw = -(-H // TILE_H), -(-W // TILE_W)

    def reduce(a, f, fill):                                   # over the in-image pixels of each tile
        p = np.full((th * TILE_H, tw * TILE_W), fill, np.int64)
        p[:H, :W] = a
        return f(f(p.reshape(th, TILE_H, tw, TILE_W), axis=3), axis=1)

    bx0 = reduce(xa, np.min, 1 << 40) & ~3                     # left edge rounded down to 16 bytes
    wx = reduce(xb, np.max, -(1 << 40)) - bx0
    wy = reduce(yb, np.max, -(1 << 40)) - reduce(ya, np.min, 1 << 40)
    tier = np.full((th, tw), len(WINDOWS), np.int64)
    for t in reversed(range(len(WINDOWS))):
        rows, cols = WINDOWS[t]
        tier[(wx < cols) & (wy < rows)] = t
    return tier


def _counts(flow):
    return tuple(int(n) for n in np.bincount(_tiers(flow).ravel(), minlength=len(TIERS)))


def _zoom(n, s):
    j = np.arange(n, dtype=np.float32)
    s, half = np.float32(s), np.float32(n / 2)
    return np.stack(np.broadcast_arrays(s * (j[None, :] - half), s * (j[:, None] - half)), -1).astype(np.float32)


def _banded(H, W):
    """Bands of 64 rows (whole tiles) that cycle through a constant flow and N(0, 1 / 2 / 5 / 40 px): every tier in one launch."""
    f = np.empty((H, W, 2), np.float32)
    f[:] = (0.37, -0.61)
    for k, sigma in enumerate((1.0, 2.0, 5.0, 40.0), 1):
        rows = (np.arange(H) // 64) % 5 == k
        f[rows] = synth.noise_flow(H, W, sigma, seed=7 + k)[rows]
    return f


@functools.lru_cache(maxsize=None)
def _flow(name):
    """The flows of the tier table, [H,W,2] float32."""
    if name == "const":
        return np.broadcast_to(np.array([0.37, -0.61], np.float32), (512, 512, 2)).copy()
    if name.startswith("noise"):
        return synth.noise_flow(1024, 1024, float(name[5:]), seed=7)
    if name.startswith("zoom"):
        return _zoom(1024, float(name[4:]))
    if name == "fold":
        return synth.random_fold_flow(2048, 2048, 555)[0]
    if name == "banded":
        return _banded(1024, 1024)
    raise KeyError(name)


# flow -> tiles per tier (small, mid, large, partial, gather)
TIER_TABLE = {
    "const": (512, 0, 0, 0, 0),
    "noise1": (113, 1935, 0, 0, 0),
    "noise2": (0, 73, 1975, 0, 0),
    "noise3": (0, 10, 1320, 718, 0),
    "noise5": (0, 0, 27, 2021, 0),
    "noise8": (0, 0, 0, 430, 1618),
    "noise40": (0, 0, 0, 0, 2048),
    "zoom0.2": (512, 1536, 0, 0, 0),
    "zoom0.4": (768, 0, 1280, 0, 0),
    "zoom1.0": (512, 512, 0, 1024, 0),
    "fold": (7865, 0, 51, 96, 180),
    "banded": (525, 381, 374, 384, 384),
}


def test_tier_mirror_pins_the_tile_paths_each_flow_reaches():
    """CPU: the flows of the GPU tests reach the tiers they are meant for, and every tier gets hundreds of tiles."""
    got = {name: _counts(_flow(name)) for name in TIER_TABLE}
    assert got == TIER_TABLE
    totals = np.sum(list(got.values()), axis=0)
    assert (totals >= 400).all(), dict(zip(TIERS, totals))
    # the config-5 section: DESIGN 4.4 reports the same 97.9 % small tiles from a GPU measurement
    fold = _counts(synth.random_fold_flow(4096, 4096, 555)[0])
    assert sum(fold) == 32768 and fold[0] == 32085


# ---------------------------------------------------------------- GPU: bit-exactness against the oracle
def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _planar(flow):
    """[B,H,W,2] numpy -> the view every reference call site passes: permute(0,2,3,1) of a planar [B,2,H,W] CUDA tensor."""
    return torch.from_numpy(np.ascontiguousarray(flow.transpose(0, 3, 1, 2))).cuda().permute(0, 2, 3, 1)


def _takes_tma(moving, flow):
    """The layout conditions under which sstem_warp_forward runs warp_torch_tma_kernel (try_launch_warp_tma)."""
    W = moving.shape[3]
    fs = flow.stride()
    return (moving.shape[1] in (1, 3) and W % 4 == 0 and fs[2] == 1 and fs[1] >= W and fs[0] % 4 == fs[1] % 4 == fs[3] % 4 == 0
            and moving.data_ptr() % 16 == 0 and flow.data_ptr() % 16 == 0)


def _moving(B, C, H, W, seed):
    """Random [0, 1) images, except a checkerboard of 16x16 blocks within half a gray level of 2/255: the stitch keeps a
    warped pixel from gray level 2 up and takes the interpolated one below, so those blocks land on both sides."""
    r = np.random.default_rng(seed)
    m = r.random((B, C, H, W), dtype=np.float32)
    near = (np.arange(H)[:, None] // 16 + np.arange(W)[None, :] // 16) % 2 == 0
    m[:, :, near] = ((2.0 + r.uniform(-0.5, 0.5, (B, C, int(near.sum())))) / 255.0).astype(np.float32)
    return m


def _assert_same(got, want, what, flows=None):
    """Bit-equal, except that a NaN only has to be a NaN (the payload of 0 * Inf differs between the CPU and the GPU).
    On a mismatch, `flows` ([B,H,W,2]) names the tiers of the tiles that differ."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, got.dtype, want.shape, want.dtype)
    if got.dtype == np.float32:
        nan = np.isnan(want)
        bad = (np.isnan(got) != nan) | (~nan & (_bits(got) != _bits(want)))
    else:
        bad = got != want
    if bad.any():
        where = ""
        if flows is not None:                                   # [B,C,H,W] or [B,H,W] -> per-tier count of differing pixels
            bad_bhw = bad.reshape(bad.shape[0], -1, *bad.shape[-2:]).any(axis=1)
            per_tier = np.zeros(len(TIERS), np.int64)
            for b in range(bad_bhw.shape[0]):
                t = np.repeat(np.repeat(_tiers(flows[b]), TILE_H, 0), TILE_W, 1)[: bad_bhw.shape[1], : bad_bhw.shape[2]]
                per_tier += np.bincount(t[bad_bhw[b]], minlength=len(TIERS))
            where = f"; pixels per tier {dict(zip(TIERS, per_tier.tolist()))}"
        first = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} values differ, first at {first}: "
                             f"got {got[first]!r}, want {want[first]!r}{where}")


def _check(moving_np, flows, seed=0):
    """SpatialTransformation through a planar flow view, and warp_and_stitch (gray and stitch), against the oracle.
    Returns the oracle's warped image and gray section."""
    from sstem_restoration_b200 import SpatialTransformation, warp_and_stitch
    B, C, H, W = moving_np.shape
    moving, flow = torch.from_numpy(moving_np).cuda(), _planar(flows)
    assert _takes_tma(moving, flow)
    want = oracle.warp_torch_restated(moving_np, flows)
    _assert_same(SpatialTransformation(True)(moving, flow).cpu().numpy(), want, "warp", flows)
    interp = np.random.default_rng(seed).integers(0, 256, (B, H, W), dtype=np.uint8)
    gray, st = warp_and_stitch(moving, flow, torch.from_numpy(interp).cuda())
    want_gray, want_st = zip(*(oracle.warp_stitch_restated(want[b], interp[b]) for b in range(B)))
    _assert_same(gray.cpu().numpy(), np.stack(want_gray), "warp_and_stitch gray", flows)
    _assert_same(st.cpu().numpy(), np.stack(want_st), "warp_and_stitch stitch", flows)
    return want, np.stack(want_gray)


TABLE_FLOWS = [n for n in TIER_TABLE if n != "banded"]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("name", TABLE_FLOWS)
def test_every_tier_is_bit_exact(name, C):
    f = _flow(name)
    H, W, _ = f.shape
    _check(_moving(1, C, H, W, seed=C), f[None], seed=C)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
def test_all_tiers_in_one_launch_and_the_stitch_threshold_in_each(C):
    """The banded flow sends tiles of every tier through one launch; in each tier's tiles the warped gray level takes
    both 1 and 2, so the stitch threshold (gray >= 2 keeps the warped pixel) is decided in every tier."""
    f = _flow("banded")
    H, W, _ = f.shape
    _, gray = _check(_moving(1, C, H, W, seed=10 + C), f[None], seed=C)
    tier = np.repeat(np.repeat(_tiers(f), TILE_H, 0), TILE_W, 1)[:H, :W]
    for t, name in enumerate(TIERS):
        g = gray[0][tier == t]
        assert (g == 1).sum() > 100 and (g == 2).sum() > 100, (name, np.bincount(g, minlength=4)[:4])


@pytest.mark.gpu
def test_config5_section_fold_at_4096():
    """1x1x4096^2 on the SFF fold flow: the warp_and_stitch call of restore_stack, and the same warp unfused."""
    f = synth.random_fold_flow(4096, 4096, 555)[0]
    _check(_moving(1, 1, 4096, 4096, seed=5), f[None], seed=5)


def _ragged_flow(kind, H, W):
    if kind == "fold":
        return synth.random_fold_flow(H, W, 555)[0]
    if kind.startswith("noise"):
        return synth.noise_flow(H, W, float(kind[5:]), seed=H + W)
    if kind == "half_out":                                     # taps straddle the 1-px zero border halfway across
        return np.broadcast_to(np.array([W / 2 + 0.3, -(H / 2) - 0.6], np.float32), (H, W, 2)).copy()
    raise KeyError(kind)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("kind", ["fold", "noise1", "noise5", "noise40"])
def test_ragged_shape_last_tile_row_and_column(kind, C):
    """H % 8 = 1 and W % 64 = 44: the last tile row holds one image row and the last tile column 44 image columns (flows
    that move the taps far from such a tile: test_taps_outside_the_image_read_the_zero_border)."""
    H, W = 1001, 1004
    _check(_moving(1, C, H, W, seed=C), _ragged_flow(kind, H, W)[None], seed=C)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("H,W", [(8, 4), (1, 4), (3, 60)])
@pytest.mark.parametrize("kind", ["noise1", "noise5", "half_out"])
def test_images_smaller_than_one_tile(H, W, kind, C):
    flows = np.stack([_ragged_flow(kind, H, W), synth.noise_flow(H, W, 1.5, seed=1)])       # a flow of its own per image
    _check(_moving(2, C, H, W, seed=H * W), flows, seed=C)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
def test_batch_entries_have_their_own_flow_and_image(C):
    """A different flow and image per batch entry (fold, N(0, 5 px), all tiers): batch coordinates of the flow and image
    tensor maps and of the global gathers."""
    n = 1024
    flows = np.stack([synth.random_fold_flow(n, n, 555)[0], synth.noise_flow(n, n, 5.0, seed=3), _flow("banded")])
    _check(_moving(3, C, n, n, seed=20 + C), flows, seed=C)


FAR = [(1e6, 0.0), (-1e6, 0.0), (0.0, 1e6), (0.0, -1e6), (3e9, -3e9), (-3e9, 3e9), (1e6, 1e6), (-1e6, -1e6)]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("H,W", [(1001, 1004), (64, 128)])
@pytest.mark.parametrize("fx,fy", FAR + [("half", "half"), ("-half", "-half")])
def test_taps_outside_the_image_read_the_zero_border(fx, fy, H, W, C):
    """Every tap off the image on one side (|x| < 2^62: beyond 2^63 the reference's float-to-int64 cast is undefined):
    small windows that lie wholly outside the image, which the TMA unit zero-fills; and half-out translations whose taps
    straddle the 1-px zero border.  A fractional part keeps all four weights nonzero."""
    if fx == "half":
        fx, fy = W / 2 + 0.3, -(H / 2) - 0.6
    elif fx == "-half":
        fx, fy = -(W / 2) - 0.7, H / 2 + 0.2
    f = np.empty((H, W, 2), np.float32)
    f[..., 0] = fx + 0.25 * (fx != 0)
    f[..., 1] = fy + 0.75 * (fy != 0)
    assert _counts(f)[0] == _tiers(f).size                    # all small windows
    _check(_moving(1, C, H, W, seed=7), f[None], seed=C)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
def test_non_finite_images(C):
    """NaN and +-Inf in the moving image, in tiles of every tier: the reference computes 0 * Inf = NaN for a zero weight
    on an infinite pixel, so NaN / Inf positions and all finite bits must match."""
    from sstem_restoration_b200 import SpatialTransformation
    f = _flow("banded")
    H, W, _ = f.shape
    m = _moving(1, C, H, W, seed=30 + C)
    flat = m.reshape(-1)
    flat[::997] = np.nan
    flat[401::1009] = np.inf
    flat[613::1013] = -np.inf
    with np.errstate(invalid="ignore"):
        want = oracle.warp_torch_restated(m, f[None])
    assert np.isnan(want).sum() > 1000 and np.isposinf(want).sum() > 100 and np.isneginf(want).sum() > 100
    got = SpatialTransformation(True)(torch.from_numpy(m).cuda(), _planar(f[None])).cpu().numpy()
    _assert_same(got, want, "warp", f[None])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["banded", "ragged_fold"])
def test_one_plane_equals_the_replicated_section(kind):
    """restore_stack warps and stitches one plane of a gray section replicated x3: that must give the bits of the C = 3 call."""
    from sstem_restoration_b200 import warp_and_stitch
    f = _flow("banded") if kind == "banded" else synth.random_fold_flow(1001, 1004, 555)[0]
    H, W, _ = f.shape
    one = torch.from_numpy(_moving(1, 1, H, W, seed=40)).cuda()
    flow = _planar(f[None])
    interp = torch.from_numpy(np.random.default_rng(41).integers(0, 256, (1, H, W), dtype=np.uint8)).cuda()
    g1, s1 = warp_and_stitch(one, flow, interp)
    g3, s3 = warp_and_stitch(one.expand(1, 3, H, W).contiguous(), flow, interp)
    assert torch.equal(g1, g3) and torch.equal(s1, s3)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["planar_view", "padded_pitch", "batch_broadcast", "interleaved", "nhwc_output",
                                    "two_channels", "moving_not_16_byte_aligned"])
def test_flow_and_image_layouts(layout):
    """One rough flow (partial and large tiers) through each layout sstem_warp_forward dispatches on: the TMA kernel where
    the tensor-map rules hold, the direct kernel otherwise; every one bit-equal to the oracle."""
    from sstem_restoration_b200 import SpatialTransformation, warp_and_stitch
    B, H, W = 2, 512, 512
    C = 2 if layout == "two_channels" else 3
    m_np = _moving(B, C, H, W, seed=50)
    f_np = np.stack([synth.noise_flow(H, W, 4.0, seed=51), synth.noise_flow(H, W, 4.0, seed=52)])
    moving = torch.from_numpy(m_np).cuda()
    if layout == "batch_broadcast":                            # batch stride 0: the tensor map encodes it or the call falls back
        f_np = np.broadcast_to(f_np[:1], f_np.shape)
        flow = _planar(f_np[:1]).expand(B, H, W, 2)
        assert flow.stride(0) == 0
    elif layout == "padded_pitch":                             # row pitch W + 8
        base = torch.zeros((B, 2, H, W + 8), device="cuda")
        base[..., :W] = torch.from_numpy(np.ascontiguousarray(f_np.transpose(0, 3, 1, 2))).cuda()
        flow = base[..., :W].permute(0, 2, 3, 1)
        assert flow.stride(1) == W + 8 and _takes_tma(moving, flow)
    elif layout == "interleaved":
        flow = torch.from_numpy(f_np).cuda()
        assert flow.is_contiguous()
    else:
        flow = _planar(f_np)
    if layout == "moving_not_16_byte_aligned":
        buf = torch.empty(moving.numel() + 1, device="cuda")
        buf[1:] = moving.reshape(-1)
        moving = buf[1:].view(B, C, H, W)
        assert moving.data_ptr() % 16 == 4
    want = oracle.warp_torch_restated(m_np, f_np)
    nhwc = layout == "nhwc_output"
    got = SpatialTransformation(True, nhwc_memory=nhwc)(moving, flow)
    if nhwc:
        assert got.permute(0, 2, 3, 1).is_contiguous()
    _assert_same(got.cpu().numpy(), want, layout, f_np)
    if C in (1, 3) and not nhwc:
        interp = np.random.default_rng(53).integers(0, 256, (B, H, W), dtype=np.uint8)
        gray, st = warp_and_stitch(moving, flow, torch.from_numpy(interp).cuda())
        want_gray, want_st = zip(*(oracle.warp_stitch_restated(want[b], interp[b]) for b in range(B)))
        _assert_same(gray.cpu().numpy(), np.stack(want_gray), layout + " gray", f_np)
        _assert_same(st.cpu().numpy(), np.stack(want_st), layout + " stitch", f_np)
