"""Quick kernel-level timing of the sepconv / warp entry points (CUDA events, inputs > L2 rotated).
Usage: python tools/bench_kernels.py [fwd] [bwd] [warp] [gi] [tiled] [gray] [tail] [tiledbwd]"""
import os
import sys
import json
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import sstem_restoration_b200 as pkg  # noqa: E402
from sstem_restoration_b200 import _lib  # noqa: E402

K = 51


def timeit(fn, reps=5, warm=2):
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


def main():
    what = set(sys.argv[1:]) or {"fwd", "bwd", "warp"}
    dev = "cuda"
    lib = _lib.load()
    peak, mhz = pkg.fp32_peak_probe()
    print(json.dumps({"fp32_probe_tflops": round(peak, 2), "probe_mhz": round(mhz)}))
    for (B, C, H, W) in [(1, 3, 256, 256), (1, 1, 256, 256), (16, 3, 512, 512), (1, 3, 2048, 2048), (1, 1, 2048, 2048)]:
        torch.manual_seed(0)
        inp = torch.rand((B, C, H + 50, W + 50), device=dev)
        v = torch.softmax(torch.randn((B, K, H, W), device=dev), 1)
        h = torch.softmax(torch.randn((B, K, H, W), device=dev), 1)
        g = torch.randn((B, C, H, W), device=dev)
        out = torch.empty((B, C, H, W), device=dev)
        st = torch.cuda.current_stream().cuda_stream
        px = B * H * W
        if "fwd" in what:
            ms = timeit(lambda: lib.sstem_sepconv_forward(inp.data_ptr(), v.data_ptr(), h.data_ptr(), out.data_ptr(), B, C, H, W, K, 0, st))
            fl = 2 * C * K * (K + 1) * px
            print(json.dumps({"op": "fwd", "shape": [B, C, H, W], "ms": round(ms, 4), "gpix_s": round(px / ms / 1e6, 3),
                              "tflops_alg": round(fl / ms / 1e9, 2), "frac_probe": round(fl / ms / 1e9 / peak, 3),
                              "tap_GBs": round(px * 408 / ms / 1e6, 1)}))
        if "bwd" in what:
            gv, gh = torch.empty_like(v), torch.empty_like(h)
            ms = timeit(lambda: lib.sstem_sepconv_backward(g.data_ptr(), inp.data_ptr(), v.data_ptr(), h.data_ptr(), None, gv.data_ptr(), gh.data_ptr(), B, C, H, W, K, 0, st), reps=3, warm=1)
            fl = 2 * (C + 2) * K * K * px
            print(json.dumps({"op": "bwd_taps", "shape": [B, C, H, W], "ms": round(ms, 4), "gpix_s": round(px / ms / 1e6, 3),
                              "tflops_alg": round(fl / ms / 1e9, 2), "frac_probe": round(fl / ms / 1e9 / peak, 3)}))
            del gv, gh
        if "tiled" in what:
            vt, ht = pkg.taps_to_tiled(v), pkg.taps_to_tiled(h)
            for flag, nm in ((0, "fwd_tiled"), (2, "fwd_tiled_gray")):
                if flag and C != 3:
                    continue
                if flag:
                    inp[:, 1:] = inp[:, :1]
                ms = timeit(lambda: lib.sstem_sepconv_forward_tiled(inp.data_ptr(), vt.data_ptr(), ht.data_ptr(), out.data_ptr(), B, C, H, W, K, flag, st))
                ms0 = timeit(lambda: lib.sstem_sepconv_forward(inp.data_ptr(), v.data_ptr(), h.data_ptr(), out.data_ptr(), B, C, H, W, K, flag, st))
                print(json.dumps({"op": nm, "shape": [B, C, H, W], "ms_tiled": round(ms, 4), "ms_nchw": round(ms0, 4),
                                  "gpix_s_tiled": round(px / ms / 1e6, 3), "tap_GBs_tiled": round(px * 408 / ms / 1e6, 1), "tap_GBs_nchw": round(px * 408 / ms0 / 1e6, 1)}))
            del vt, ht
        if "tiledbwd" in what and C == 3 and (B, H, W) in ((16, 512, 512), (1, 2048, 2048)):
            # tap gradients on tile-major taps vs [B,51,H,W], general and gray x3; then the tail's tap gradients (both frames)
            vt, ht = pkg.taps_to_tiled(v), pkg.taps_to_tiled(h)
            gv, gh, gvt, ght = torch.empty_like(v), torch.empty_like(h), torch.empty_like(vt), torch.empty_like(ht)
            res = {"op": "tiledbwd", "shape": [B, C, H, W]}
            for flag, nm in ((0, "general"), (2, "gray")):
                if flag:
                    inp[:, 1:] = inp[:, :1]
                res["ms_tiled_" + nm] = round(timeit(lambda: lib.sstem_sepconv_backward_tiled(
                    g.data_ptr(), inp.data_ptr(), vt.data_ptr(), ht.data_ptr(), None, gvt.data_ptr(), ght.data_ptr(), B, C, H, W, K, flag, st), reps=3, warm=1), 4)
                res["ms_nchw_" + nm] = round(timeit(lambda: lib.sstem_sepconv_backward(
                    g.data_ptr(), inp.data_ptr(), v.data_ptr(), h.data_ptr(), None, gv.data_ptr(), gh.data_ptr(), B, C, H, W, K, flag, st), reps=3, warm=1), 4)
            f1, f2 = (torch.rand((B, 3, H, W), device=dev) for _ in range(2))
            p1, p2 = pkg.frame_mean_pad(f1), pkg.frame_mean_pad(f2)
            go = torch.rand((B, 1, H, W), device=dev) - 0.5
            gts = [torch.empty_like(vt) for _ in range(4)]
            gns = [torch.empty_like(v) for _ in range(4)]

            def tail_tiled():                              # what ModuleInterpolationTailTiled's backward launches
                for p, t in ((p2, gts[2:]), (p1, gts[:2])):
                    lib.sstem_sepconv_backward_tiled(go.data_ptr(), p.data_ptr(), vt.data_ptr(), ht.data_ptr(), None, t[0].data_ptr(), t[1].data_ptr(),
                                                     B, 1, H, W, K, 0, st)
            res["ms_tail_bwd_tiled"] = round(timeit(tail_tiled, reps=3, warm=1), 4)
            res["ms_tail_bwd_nchw"] = round(timeit(lambda: lib.sstem_interp_tail_backward(
                go.data_ptr(), f1.data_ptr(), f2.data_ptr(), 3 * H * W, v.data_ptr(), h.data_ptr(), v.data_ptr(), h.data_ptr(),
                *[t.data_ptr() for t in gns], B, 3, H, W, K, 0, st), reps=3, warm=1), 4)
            print(json.dumps(res))
            del vt, ht, gv, gh, gvt, ght, f1, f2, p1, p2, go, gts, gns
        if "gray" in what and C == 3:
            gv, gh = torch.empty_like(v), torch.empty_like(h)
            inp[:, 1:] = inp[:, :1]
            ms_f = timeit(lambda: lib.sstem_sepconv_forward(inp.data_ptr(), v.data_ptr(), h.data_ptr(), out.data_ptr(), B, C, H, W, K, 2, st))
            ms_b = timeit(lambda: lib.sstem_sepconv_backward(g.data_ptr(), inp.data_ptr(), v.data_ptr(), h.data_ptr(), None, gv.data_ptr(), gh.data_ptr(), B, C, H, W, K, 2, st), reps=3, warm=1)
            print(json.dumps({"op": "gray_x3 fwd / bwd_taps", "shape": [B, C, H, W], "ms_fwd": round(ms_f, 4), "ms_bwd": round(ms_b, 4),
                              "fwd_gpix_s": round(px / ms_f / 1e6, 3), "bwd_gpix_s": round(px / ms_b / 1e6, 3),
                              "fwd_tapGBs": round(px * 408 / ms_f / 1e6, 1), "bwd_GBs": round(px * 840 / ms_b / 1e6, 1)}))
            del gv, gh
        if "tail" in what and C == 3:
            # fused interpolation tail vs the unfused expression it replaces (model_interp.py:90-97)
            f1, f2 = torch.rand((B, 1, H, W), device=dev).expand(B, 3, H, W).contiguous(), torch.rand((B, 1, H, W), device=dev).expand(B, 3, H, W).contiguous()
            v2, h2 = torch.softmax(torch.randn((B, K, H, W), device=dev), 1), torch.softmax(torch.randn((B, K, H, W), device=dev), 1)
            pad = torch.nn.ReplicationPad2d(25)

            def unfused():
                y = pkg.SeparableConvolution.apply(pad(f2), v2, h2) + pkg.SeparableConvolution.apply(pad(f1), v, h)
                return torch.mean(y, dim=1, keepdim=True)
            res = {"op": "interp_tail", "shape": [B, C, H, W], "ms_unfused": round(timeit(unfused), 4)}
            for mode in ("off", "assert"):
                pkg.set_gray_replicated(mode)
                ms = timeit(lambda: pkg.interpolation_tail(f1, f2, v, h, v2, h2))
                res["ms_fused_gray_" + mode] = round(ms, 4)
                res["gpix_s_gray_" + mode] = round(px / ms / 1e6, 3)
                res["tapGBs_gray_" + mode] = round(px * 816 / ms / 1e6, 1)
            pkg.set_gray_replicated("off")
            gvs = [torch.empty_like(v) for _ in range(4)]
            go = torch.randn((B, 1, H, W), device=dev)
            for flag in (0, 2):
                ms = timeit(lambda: lib.sstem_interp_tail_backward(go.data_ptr(), f1.data_ptr(), f2.data_ptr(), 3 * H * W, v.data_ptr(), h.data_ptr(), v2.data_ptr(), h2.data_ptr(),
                                                                   *[t.data_ptr() for t in gvs], B, C, H, W, K, flag, st), reps=3, warm=1)
                res["ms_bwd_flag%d" % flag] = round(ms, 4)
            print(json.dumps(res))
            del f1, f2, v2, h2, gvs, go
        if "gi" in what:
            gi = torch.empty_like(inp)
            ms = timeit(lambda: lib.sstem_sepconv_backward(g.data_ptr(), inp.data_ptr(), v.data_ptr(), h.data_ptr(), gi.data_ptr(), None, None, B, C, H, W, K, 0, st), reps=2, warm=1)
            fl = 2 * C * K * (K + 1) * px
            print(json.dumps({"op": "bwd_input", "shape": [B, C, H, W], "ms": round(ms, 4), "gpix_s": round(px / ms / 1e6, 3), "tflops_alg": round(fl / ms / 1e9, 2), "frac_probe": round(fl / ms / 1e9 / peak, 3)}))
        del inp, v, h, g, out
        torch.cuda.empty_cache()
    if "warp" in what:
        st = pkg.SpatialTransformation(True)
        for (B, C, H, W) in [(1, 3, 2048, 2048), (1, 3, 4096, 4096), (1, 1, 4096, 4096)]:
            n = max(2, int(1.0e9 // (B * H * W * (8 * C + 8))))
            sets = [(torch.rand((B, C, H, W), device=dev), (5 * torch.randn((B, 2, H, W), device=dev)).permute(0, 2, 3, 1)) for _ in range(n)]
            smooth = [(a, (torch.zeros((B, 2, H, W), device=dev) + 3.3).permute(0, 2, 3, 1)) for a, _ in sets]
            for name, ss in (("noise5px", sets), ("const3.3px", smooth)):
                ms = timeit(lambda: [st(a, f) for a, f in ss]) / n
                print(json.dumps({"op": "warp_" + name, "shape": [B, C, H, W], "ms": round(ms, 5), "GBs": round(B * H * W * (8 * C + 8) / ms / 1e6, 1),
                                  "gpix_s": round(B * H * W / ms / 1e6, 2)}))
            del sets, smooth
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
