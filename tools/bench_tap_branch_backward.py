"""Timing of the tap branch backward: the three half-resolution Conv2d -> ReLU layers of IFNet._kernel_module on
branch_conv3x3_backward (per layer and chained), and one training step of ModuleTapBranch(trainable=True), next to torch's
TF32 autograd of the same layers (cuDNN, cudnn.benchmark).  CUDA events, inputs rotated through more than the 126 MB L2.

Shapes (x): [16,64,256,256] (the training batch), [1,64,1024,1024], [1,64,2048,2048].  Per layer the public entry point
is timed asking for one gradient at a time; the mask / convert step is the call that asks for grad_bias alone (mask
kernel + a 64-part sum), and grad_x, grad_weight + grad_bias are that call's time subtracted from theirs.  Useful TFLOP/s
of the weight gradient count 2 * B * h * w * cin * cout * 9; the share of peak uses 837.9 TFLOP/s, the measured TF32
denominator of DESIGN 4.11.

    python tools/bench_tap_branch_backward.py [--reps 10] [--out profiles/tap_branch_backward_b200.jsonl]

Prints and writes one JSON line per measurement, the first naming the card, its power limit and max SM clock."""
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
    ap.add_argument("--shapes", default="16x256,1x1024,1x2048", help="comma-separated BxS for x [B,64,S,S]")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles",
                                                  "tap_branch_backward_b200.jsonl"))
    a = ap.parse_args()
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(json.dumps(d))

    emit({"card": card()})
    nn = torch.nn
    torch.backends.cudnn.allow_tf32 = True                 # torch's default for convolutions
    torch.backends.cudnn.benchmark = True
    for spec in a.shapes.split(","):
        B, h = (int(v) for v in spec.split("x"))
        shape = [B, 64, h, h]
        torch.manual_seed(0)
        seq = nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(), nn.Conv2d(64, 51, 3, 1, 1),
                            nn.ReLU(), nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True), nn.Conv2d(51, 51, 3, 1, 1)).cuda()
        m = pkg.ModuleTapBranch(tiled=False, trainable=True).cuda()
        m.load_state_dict(seq.state_dict())
        layers = [getattr(m, k) for k in ("0", "2", "4")]
        packed = [pkg.pack_branch_conv_weight(l.weight.detach()) for l in layers]
        adj = [pkg.pack_branch_conv_weight_adjoint(l.weight.detach()) for l in layers]
        dims = [(64, 64), (64, 64), (64, 51)]              # (cin, cout)
        xs = [torch.relu(torch.randn(shape, device="cuda")) for _ in range(2)]   # >= 256 MB each: beyond L2
        it = [0]

        def nxt(lst):
            it[0] += 1
            return lst[it[0] % len(lst)]

        def report(op, fn, flop=None, **extra):
            ms = timeit(fn, a.reps)
            d = {"op": op, "x": shape, "ms": round(ms, 4)}
            if flop:
                d["useful_tflops"] = round(flop / ms / 1e9, 1)
                d["share_of_tf32_peak"] = round(flop / ms / 1e9 / TF32_PEAK, 3)
            d.update(extra)
            emit(d)
            return ms

        with torch.no_grad():
            # per rotated input: the forward's activations in the layouts the module keeps, and a gradient per layer output
            acts = []
            for x in xs:
                a1 = pkg.branch_conv3x3(x, packed[0], layers[0].bias, chunked_out=True)
                a2 = pkg.branch_conv3x3(a1, packed[1], layers[1].bias, chunked_in=True, chunked_out=True)
                a3 = pkg.branch_conv3x3(a2, packed[2], layers[2].bias, chunked_in=True)
                acts.append((x, a1, a2, a3))
            gouts = [[torch.randn((B, c, h, h), device="cuda") for _, c in dims] for _ in xs]
            px = B * h * h
            layer_ms = []
            for L in range(3):
                cin, cout = dims[L]
                ci, co = L > 0, L < 2

                def call(need, L=L, cin=cin, cout=cout, ci=ci, co=co):
                    k = it[0] = it[0] + 1
                    act, g = acts[k % len(acts)], gouts[k % len(gouts)][L]
                    return pkg.branch_conv3x3_backward(g, act[L + 1], act[L], adj[L] if need[0] else None, cin, cout,
                                                       chunked_in=ci, chunked_out=co, need=need)

                name = f"layer{L}_{cin}to{cout}"
                t_b = report(f"{name}_mask_convert", lambda: call((False, False, True)), how="call asking for grad_bias alone")
                t_x = report(f"{name}_grad_x_call", lambda: call((True, False, False)), 2 * px * cin * cout * 9)
                t_w = report(f"{name}_grad_weight_bias_call", lambda: call((False, True, True)), 2 * px * cin * cout * 9)
                t_all = report(f"{name}_whole_layer_backward", lambda: call((True, True, True)), 2 * 2 * px * cin * cout * 9)
                emit({"op": f"{name}_grad_x", "x": shape, "ms": round(t_x - t_b, 4), "how": "grad_x call minus mask call"})
                fw = 2 * px * cin * cout * 9
                emit({"op": f"{name}_grad_weight_bias", "x": shape, "ms": round(t_w - t_b, 4), "how": "grad_weight+bias call minus mask call",
                      "useful_tflops": round(fw / (t_w - t_b) / 1e9, 1), "share_of_tf32_peak": round(fw / (t_w - t_b) / 1e9 / TF32_PEAK, 3)})
                layer_ms.append(t_all)

            def ours_three():
                k = it[0] = it[0] + 1
                x, a1, a2, a3 = acts[k % len(acts)]
                g = gouts[k % len(gouts)][2]
                g, _, _ = pkg.branch_conv3x3_backward(g, a3, a2, adj[2], 64, 51, chunked_in=True)
                g, _, _ = pkg.branch_conv3x3_backward(g, a2, a1, adj[1], 64, 64, chunked_in=True, chunked_out=True)
                pkg.branch_conv3x3_backward(g, a1, x, adj[0], 64, 64, chunked_out=True)
            flop3 = 2 * 2 * px * 9 * (64 * 64 * 2 + 64 * 51)
            t_ours = report("three_conv_backward", ours_three, flop3, how="branch_conv3x3_backward x 3, all gradients")

        # torch: the same three Conv2d -> ReLU layers, TF32 autograd, graph built once per rotated input
        tin = [x.clone().requires_grad_(True) for x in xs]
        touts = [seq[5](seq[4](seq[3](seq[2](seq[1](seq[0](x)))))) for x in tin]
        params3 = [p for i in (0, 2, 4) for p in seq[i].parameters()]

        def torch_three():
            k = it[0] = it[0] + 1
            torch.autograd.grad(touts[k % 2], [tin[k % 2]] + params3, gouts[k % len(gouts)][2], retain_graph=True)
        t_torch = report("torch_three_conv_backward_tf32", torch_three, flop3)
        emit({"op": "three_conv_backward_speedup", "x": shape, "ours_ms": round(t_ours, 4), "torch_ms": round(t_torch, 4),
              "speedup": round(t_torch / t_ours, 2)})
        del touts, tin

        # one training step (forward + backward, x requires grad) of the whole branch
        full_g = torch.randn((B, 51, 2 * h, 2 * h), device="cuda")
        xr = [x.clone().requires_grad_(True) for x in xs]

        def step(mod):
            def f():
                k = it[0] = it[0] + 1
                mod(xr[k % 2]).backward(full_g)
            return f
        t_ms = report("module_tap_branch_training_step", step(m), how="ModuleTapBranch(tiled=False, trainable=True)")
        t_ts = report("torch_sequential_training_step_tf32", step(seq))
        emit({"op": "training_step_speedup", "x": shape, "ours_ms": round(t_ms, 4), "torch_ms": round(t_ts, 4),
              "speedup": round(t_ts / t_ms, 2)})
        del xs, acts, gouts, xr, full_g, m, seq
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
