"""fp64 restatement of the backward of the tap producer, y = conv3x3(up(x), W) + b (oracle.tap_conv3x3_restated):

    grad_x      = up^T(conv3x3(gy, W')),  W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]
    grad_weight = sum over pixels of gy x up(x), zero padded by 1 and shifted per tap
    grad_bias   = sum of gy over pixels

up is written as two interpolation matrices, Ry [H, h] and Rx [W, w], with the float32 index and weight expressions of
oracle.upsample2x_align_corners_restated (ATen's), so up(x) = Ry x Rx^T and up^T(g) = Ry^T g Rx exactly."""
import numpy as np

import oracle


def upsample_axis_matrix(n_in, n_out):
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0)
    r = (scale * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = r.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    l1 = (r - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1) - l1).astype(np.float32)
    m = np.zeros((n_out, n_in))
    np.add.at(m, (np.arange(n_out), i0), l0.astype(np.float64))
    np.add.at(m, (np.arange(n_out), i1), l1.astype(np.float64))
    return m


def upsample2x(x):
    x = np.asarray(x, np.float64)
    h, w = x.shape[2:]
    return np.einsum("Yi,bcij,Xj->bcYX", upsample_axis_matrix(h, 2 * h), x, upsample_axis_matrix(w, 2 * w), optimize=True)


def upsample2x_adjoint(g):
    g = np.asarray(g, np.float64)
    H, W = g.shape[2:]
    return np.einsum("Yi,bcYX,Xj->bcij", upsample_axis_matrix(H // 2, H), g, upsample_axis_matrix(W // 2, W), optimize=True)


def adjoint_weight(weight):
    """W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]"""
    return np.ascontiguousarray(np.asarray(weight).transpose(1, 0, 2, 3)[:, :, ::-1, ::-1])


def tap_conv3x3_backward_restated(gy, x, weight, upsample=True):
    """(grad_x, grad_weight, grad_bias) in fp64; gy [B,cout,H,W], x [B,cin,h,w], weight [cout,cin,3,3]."""
    gy = np.asarray(gy, np.float64)
    gU = oracle.tap_conv3x3_restated(gy, adjoint_weight(weight), None, upsample=False)
    gx = upsample2x_adjoint(gU) if upsample else gU
    up = upsample2x(x) if upsample else np.asarray(x, np.float64)
    B, C, H, W = up.shape
    pad = np.zeros((B, C, H + 2, W + 2))
    pad[:, :, 1:-1, 1:-1] = up
    gw = np.zeros((gy.shape[1], C, 3, 3))
    for dy in range(3):
        for dx in range(3):
            gw[:, :, dy, dx] = np.einsum("bohw,bihw->oi", gy, pad[:, :, dy:dy + H, dx:dx + W], optimize=True)
    return gx, gw, gy.sum(axis=(0, 2, 3))
