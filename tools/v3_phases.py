"""Where the warp time of the generation-3 sepconv kernels goes, phase by phase, at 16x3x512x512.

    python -c "from sstem_restoration_b200 import _build; _build.build(force=True, lib_path='/tmp/lib_phases.so', extra=['-DSSTEM_V3_PHASES'])"
    SSTEM_LIB_PATH=/tmp/lib_phases.so python tools/v3_phases.py

Needs a library built with -DSSTEM_V3_PHASES (the shipped build has no phase clocks).  Every warp of the forward and the
tap-gradient kernels adds the clock64 ticks it spends in each phase of its tiles; this prints each phase's share of the
summed warp time (the time before a warp's first tile and after its last is not counted):
    start    wait for the tile's horizontal taps (and upstream gradient), copy them to registers, draw the ticket
    first    the leading groups with rows still joining (forward 0-1, tap gradients 0) and the tap-buffer refill
    steady   the runtime loop over groups in which every row is active
    last     the trailing groups with rows leaving
    store    the epilogue: the forward's output, the tap gradients' grad_horizontal (grad_vertical leaves step by step
             inside the groups)
    barrier  the per-tile CTA barrier and the next ticket
"""
import ctypes
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from sstem_restoration_b200 import _lib  # noqa: E402

K = 51
PHASES = ("start", "first", "steady", "last", "store", "barrier")


def main():
    lib = _lib.load()
    for fn in ("sstem_v3_phases_fwd", "sstem_v3_phases_bwd"):
        if not hasattr(lib, fn):
            raise SystemExit(f"{_lib.LIB_PATH} has no {fn}: build it with -DSSTEM_V3_PHASES")
        getattr(lib, fn).argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]
        getattr(lib, fn).restype = ctypes.c_int
    B, C, H, W, reps = 16, 3, 512, 512, 5
    dev = "cuda"
    torch.manual_seed(0)
    inp = torch.rand((B, C, H + 50, W + 50), device=dev)
    v = torch.softmax(torch.randn((B, K, H, W), device=dev), 1)
    h = torch.softmax(torch.randn((B, K, H, W), device=dev), 1)
    g = torch.randn((B, C, H, W), device=dev)
    out, gv, gh = torch.empty_like(g), torch.empty_like(v), torch.empty_like(h)
    st = torch.cuda.current_stream().cuda_stream
    ops = {
        "fwd": ("sstem_v3_phases_fwd", lambda: lib.sstem_sepconv_forward(inp.data_ptr(), v.data_ptr(), h.data_ptr(), out.data_ptr(), B, C, H, W, K, 0, st)),
        "bwd_taps": ("sstem_v3_phases_bwd", lambda: lib.sstem_sepconv_backward(g.data_ptr(), inp.data_ptr(), v.data_ptr(), h.data_ptr(), None,
                                                                             gv.data_ptr(), gh.data_ptr(), B, C, H, W, K, 0, st)),
    }
    buf = (ctypes.c_ulonglong * len(PHASES))()
    print(f"| kernel | {' | '.join(PHASES)} | Gticks |")
    print(f"|---|{'---|' * len(PHASES)}---|")
    for name, (fn, run) in ops.items():
        run()                                              # warm-up launch
        torch.cuda.synchronize()
        assert getattr(lib, fn)(buf, 1) == 0
        for _ in range(reps):
            rc = run()
            assert rc == 0, rc
        torch.cuda.synchronize()
        assert getattr(lib, fn)(buf, 1) == 0
        ticks = [int(x) for x in buf]
        total = sum(ticks)
        assert total > 0, f"{name}: no phase ticks (did the persistent kernel run?)"
        print(f"| {name} | {' | '.join(f'{100.0 * t / total:.1f} %' for t in ticks)} | {total / reps / 1e9:.2f} |")
        print(json.dumps({"op": name, "shape": [B, C, H, W], "lib": os.path.basename(_lib.LIB_PATH),
                          "ticks_per_launch": {p: t // reps for p, t in zip(PHASES, ticks)}}), file=sys.stderr)


if __name__ == "__main__":
    main()
