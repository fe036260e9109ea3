"""A/B harness for compile-time kernel variants.

    python tools/ab.py build  MINB1=-DSSTEM_BWD3_MINB=1 PHASES=-DSSTEM_V3_PHASES                      # here (no GPU): nvcc
    gpurun -- 'python tools/ab.py run fwd bwd tail'                                                       # on the GPU box

`build` compiles one extra copy of the library per NAME into gpurun_scratch/lib_NAME.so (they travel to the GPU box with
the snapshot; gpurun_scratch/ is git-ignored).  `run` times tools/bench_kernels.py <ops> with the in-tree library
("base") and with every gpurun_scratch/lib_*.so (through SSTEM_LIB_PATH), and prints one line per variant and op at
16x3x512x512 so that the variants can be compared from a single call.
"""
import glob
import json
import os
import subprocess
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
SCRATCH = os.path.join(ROOT, "gpurun_scratch")
sys.path.insert(0, ROOT)


def build(specs):
    from sstem_restoration_b200 import _build
    os.makedirs(SCRATCH, exist_ok=True)
    for spec in specs:
        name, _, flags = spec.partition("=")
        path = os.path.join(SCRATCH, f"lib_{name}.so")
        _build.build(force=True, lib_path=path, extra=flags.split())
        print("built", path, flags)


def run(ops):
    variants = [("base", None)] + [(os.path.basename(p)[4:-3], p) for p in sorted(glob.glob(os.path.join(SCRATCH, "lib_*.so")))]
    for name, path in variants:
        env = dict(os.environ)
        if path:
            env["SSTEM_LIB_PATH"] = path
        out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_kernels.py")] + ops, env=env,
                             capture_output=True, text=True).stdout
        for line in out.splitlines():
            try:
                d = json.loads(line)
            except ValueError:
                continue
            if d.get("shape") == [16, 3, 512, 512]:
                keep = {k: v for k, v in d.items() if k.startswith("ms") or k in ("op", "frac_probe")}
                print(f"{name:>12}", json.dumps(keep))


if __name__ == "__main__":
    if len(sys.argv) < 2 or sys.argv[1] not in ("build", "run"):
        raise SystemExit(__doc__)
    (build if sys.argv[1] == "build" else run)(sys.argv[2:])
