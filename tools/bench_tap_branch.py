"""Timing of a whole tap branch (IFNet._kernel_module: three half-resolution Conv2d -> ReLU layers, upsample x2, Conv2d(51, 51,
3)) on branch_conv3x3 + the tap producer (ModuleTapBranch), layer by layer, next to torch's nn.Sequential of the same eight
layers (cuDNN, default TF32) followed by taps_to_tiled.  CUDA events, inputs rotated through more than the 126 MB L2.

Shapes (x): [1,64,1024,1024] (2048^2 taps), [1,64,2048,2048] (one 4096^2 section), [16,64,256,256] (the training batch).
Useful TFLOP/s count 2 * B * h * w * cin * cout * 9 per conv; the share of peak uses 837.9 TFLOP/s, the measured TF32
denominator of DESIGN 4.11.

    python tools/bench_tap_branch.py [--reps 10] [--out profiles/tap_branch_b200.jsonl]

Prints and writes one JSON line per measurement, the first naming the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import sstem_restoration_b200 as pkg  # noqa: E402

TF32_PEAK = 837.9


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
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
    except Exception as e:                                 # the timings still name the device
        return f"{torch.cuda.get_device_name(0)}, power limit unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "tap_branch_b200.jsonl"))
    a = ap.parse_args()
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    emit({"card": card()})
    nn = torch.nn
    torch.backends.cudnn.allow_tf32 = True                 # torch's default for convolutions
    torch.backends.cudnn.benchmark = True
    for B, h in ((1, 1024), (1, 2048), (16, 256)):
        torch.manual_seed(0)
        shape = [B, 64, h, h]
        xs = [torch.relu(torch.randn(shape, device="cuda")) for _ in range(2)]   # >= 256 MB each: beyond L2
        seq = nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 51, 3, 1, 1),
                            nn.ReLU(), nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True), nn.Conv2d(51, 51, 3, 1, 1)).cuda()
        m = pkg.ModuleTapBranch().cuda()
        m.load_state_dict(seq.state_dict())
        layers = [getattr(m, k) for k in ("0", "2", "4")]
        packed = [pkg.pack_branch_conv_weight(l.weight.detach()) for l in layers]
        it = [0]

        def nxt(lst):
            it[0] += 1
            return lst[it[0] % len(lst)]

        with torch.no_grad():
            # inputs of each layer, rotated: chunk-major activations as the module passes them
            a1 = [pkg.branch_conv3x3(x, packed[0], layers[0].bias, chunked_out=True) for x in xs]
            a2 = [pkg.branch_conv3x3(t, packed[1], layers[1].bias, chunked_in=True, chunked_out=True) for t in a1]
            a3 = [pkg.branch_conv3x3(t, packed[2], layers[2].bias, chunked_in=True) for t in a2]

            def report(op, fn, flop=None, **extra):
                ms = timeit(fn, a.reps)
                d = {"op": op, "x": shape, "ms": round(ms, 4)}
                if flop:
                    d["useful_tflops"] = round(flop / ms / 1e9, 1)
                    d["share_of_tf32_peak"] = round(flop / ms / 1e9 / TF32_PEAK, 3)
                d.update(extra)
                emit(d)
                return ms

            px = B * h * h
            f64, f51 = 2 * px * 64 * 64 * 9, 2 * px * 64 * 51 * 9
            fprod = 2 * 4 * px * 51 * 51 * 9
            t = {}
            t["conv0_nchw_in"] = report("branch_conv0_nchw_in_chunked_out", lambda: pkg.branch_conv3x3(nxt(xs), packed[0], layers[0].bias, chunked_out=True), f64)
            t["conv0"] = report("branch_conv0_chunked_in_chunked_out", lambda: pkg.branch_conv3x3(nxt(a1), packed[0], layers[0].bias, chunked_in=True, chunked_out=True), f64)
            t["conv1"] = report("branch_conv1_chunked_in_chunked_out", lambda: pkg.branch_conv3x3(nxt(a1), packed[1], layers[1].bias, chunked_in=True, chunked_out=True), f64)
            t["conv2"] = report("branch_conv2_chunked_in_nchw_out", lambda: pkg.branch_conv3x3(nxt(a2), packed[2], layers[2].bias, chunked_in=True), f51)
            t["producer"] = report("tap_producer_tiled", lambda: m._modules["7"](nxt(a3)), fprod)
            conv_ms = t["conv0_nchw_in"] - t["conv0"]
            t["branch"] = report("module_tap_branch", lambda: m(nxt(xs)), 2 * f64 + f51 + fprod)
            emit({"op": "nchw_to_chunked_conversion", "x": shape, "ms": round(conv_ms, 4),
                  "how": "conv0 with NCHW input minus conv0 with chunk-major input",
                  "share_of_branch": round(conv_ms / t["branch"], 3)})
            # torch: the same eight layers (cuDNN TF32), then the tile-major conversion the consumer needs
            t["torch"] = report("torch_sequential_tf32_plus_taps_to_tiled", lambda: pkg.taps_to_tiled(seq(nxt(xs))), 2 * f64 + f51 + fprod)
            report("torch_conv0_relu_tf32", lambda: torch.relu(seq[0](nxt(xs))), f64)
            t51 = [torch.relu(seq[4](seq[3](seq[2](seq[1](seq[0](x)))))) for x in xs]
            report("torch_conv2_relu_tf32", lambda: torch.relu(seq[4](nxt(xs))), f51)
            report("torch_upsample_conv_tf32", lambda: seq[7](seq[6](nxt(t51))), fprod)
            if h == 2048:
                emit({"op": "four_branches_per_4096_target", "x": shape, "ms_branch": round(4 * t["branch"], 3),
                      "ms_torch": round(4 * t["torch"], 3), "speedup": round(t["torch"] / t["branch"], 2)})
            del xs, a1, a2, a3, t51
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
