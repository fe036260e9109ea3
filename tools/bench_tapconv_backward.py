"""Timing of the tap producer's backward (sstem_tap_conv3x3_backward: grad_x, grad_weight, grad_bias) next to torch's own
TF32 autograd of the same layer pair (F.interpolate -> conv2d, cuDNN, allow_tf32), CUDA events, inputs rotated through
more than the 126 MB L2.  Shapes: the training step's x [16,51,256,256] and x [1,51,1024,1024] (output 512^2 / 2048^2).

    python tools/bench_tapconv_backward.py [--reps 10]

Prints the card and its power limit, then one JSON line per variant (ms per backward)."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import sstem_restoration_b200 as pkg  # noqa: E402
from sstem_restoration_b200 import _lib  # noqa: E402


def timeit(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
    except Exception as e:                                 # the timings still name the device
        q = f"{torch.cuda.get_device_name(0)}, power limit unknown ({e})"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    dev = "cuda"
    print(json.dumps({"card": card()}), flush=True)
    lib = _lib.load()
    for B, h in ((16, 256), (1, 1024)):
        H = W = 2 * h
        nrot = 2 if B > 1 else 3
        torch.manual_seed(0)
        xs = [torch.relu(torch.randn((B, 51, h, h), device=dev)) for _ in range(nrot)]
        gys = [torch.randn((B, 51, H, W), device=dev) for _ in range(nrot)]
        gts = [pkg.taps_to_tiled(g) for g in gys]
        conv = torch.nn.Conv2d(51, 51, 3, 1, 1).to(dev)
        adj = pkg.pack_tap_conv_weight_adjoint(conv.weight.detach())
        gx = torch.empty_like(xs[0])
        gw = torch.empty_like(conv.weight)
        gb = torch.empty_like(conv.bias)
        it = [0]
        stream = torch.cuda.current_stream().cuda_stream

        def ours(tiled, want_x=True, want_w=True):
            def run():
                it[0] += 1
                k = it[0] % nrot
                g = gts[k] if tiled else gys[k]
                flags = _lib.TAPCONV_UPSAMPLE2X | (_lib.TAPCONV_TILED if tiled else 0)
                code = lib.sstem_tap_conv3x3_backward(g.data_ptr(), xs[k].data_ptr(), adj.data_ptr(),
                                                      gx.data_ptr() if want_x else None, gw.data_ptr() if want_w else None,
                                                      gb.data_ptr() if want_w else None, B, 51, 51, h, h, flags, stream)
                _lib.check(code, "sstem_tap_conv3x3_backward")
            return run

        def report(name, fn):
            ms = timeit(fn, a.reps)
            print(json.dumps({"op": name, "x": [B, 51, h, h], "ms": round(ms, 4)}), flush=True)

        report("tapconv_backward_all_nchw", ours(False))
        report("tapconv_backward_all_tiled", ours(True))
        report("tapconv_backward_grad_x_only", ours(False, want_w=False))
        report("tapconv_backward_grad_w_b_only", ours(False, want_x=False))
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cudnn.benchmark = True
        graphs = []
        for x in xs:
            tx = x.clone().requires_grad_(True)
            y = conv(torch.nn.functional.interpolate(tx, scale_factor=2, mode="bilinear", align_corners=True))
            graphs.append((y, tx))

        def lib_bwd():
            it[0] += 1
            k = it[0] % nrot
            y, tx = graphs[k]
            torch.autograd.grad(y, (tx, conv.weight, conv.bias), gys[k], retain_graph=True)
        report("library_upsample_conv_tf32_backward", lib_bwd)
        del graphs, xs, gys, gts


if __name__ == "__main__":
    main()
