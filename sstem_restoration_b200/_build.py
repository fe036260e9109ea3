"""Builds libsstem_b200.so in-tree with nvcc for sm_100a (no torch headers, no JIT cache).

The library is the whole product: there is no CPU or PyTorch fallback.  Replaces the
reference's `libs/sepconv/install.bash:14-18` (nvcc for compute_37) and
`install.py:23-37` (torch.utils.ffi.create_extension).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libsstem_b200.so")
# (source, extra defines, object suffix).  The tuned sepconv kernels are ~130 template
# instantiations; they are spread over several translation units (and the tap-gradient file
# is compiled four times, one -DSSTEM_BWD_PART each) so that a build is parallel.
UNITS = [
    ("abi.cu", [], ""),
    ("sepconv_generic.cu", [], ""),
    ("sepconv_k51_fwd.cu", [], ""),
    ("sepconv_k51_bwd.cu", ["-DSSTEM_BWD_PART=0"], "_p0"),
    ("sepconv_k51_bwd.cu", ["-DSSTEM_BWD_PART=1"], "_p1"),
    ("sepconv_k51_bwd.cu", ["-DSSTEM_BWD_PART=2"], "_p2"),
    ("sepconv_k51_bwd.cu", ["-DSSTEM_BWD_PART=3"], "_p3"),
    ("sepconv_k51_bwd3.cu", [], ""),
    ("sepconv_k51_fwd3.cu", [], ""),
    ("sepconv_layout.cu", [], ""),
    ("sepconv_k51_gi.cu", [], ""),
    ("sepconv_k51_tail.cu", [], ""),
    ("warp.cu", [], ""),
    ("tapconv.cu", [], ""),
    ("sff_sim.cu", [], ""),
    ("stack_io.cu", [], ""),
    ("probe.cu", [], ""),
]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libsstem_b200.so cannot be built")


def needs_build(lib_path: str = LIB_PATH) -> bool:
    if not os.path.exists(lib_path):
        return True
    t = os.path.getmtime(lib_path)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "sstem_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False, lib_path: str = LIB_PATH, extra=None) -> str:
    """Compile every CUDA source (in parallel) and link one shared library; returns its path.

    `extra` / $SSTEM_NVCC_EXTRA: additional nvcc flags for kernel-tuning experiments
    (e.g. -DSSTEM_BWD3_MINB=1), normally together with another `lib_path`."""
    if not force and not needs_build(lib_path):
        return lib_path
    from concurrent.futures import ThreadPoolExecutor

    nvcc = _nvcc()
    extra = list(extra or []) + os.environ.get("SSTEM_NVCC_EXTRA", "").split()
    objdir = tempfile.mkdtemp(prefix="sstem_obj_")

    def compile_one(unit):
        src, defs, suffix = unit
        obj = os.path.join(objdir, os.path.splitext(src)[0] + suffix + ".o")
        cmd = [nvcc] + NVCC_FLAGS + defs + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        return obj, " ".join(cmd) + "\n" + proc.stdout + proc.stderr, proc.returncode

    try:
        with ThreadPoolExecutor(max_workers=min(len(UNITS), os.cpu_count() or 4)) as pool:
            results = list(pool.map(compile_one, UNITS))
        log = "".join(r[1] for r in results)
        failed = [r for r in results if r[2] != 0]
        if not failed:
            cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path + ".tmp"] + [r[0] for r in results]
            proc = subprocess.run(cmd, capture_output=True, text=True)
            log += " ".join(cmd) + "\n" + proc.stdout + proc.stderr
            if proc.returncode != 0:
                failed = [(None, proc.stdout + proc.stderr, proc.returncode)]
        if lib_path == LIB_PATH:
            with open(os.path.join(HERE, "build.log"), "w") as f:
                f.write(log)
        if failed:
            raise RuntimeError("nvcc failed:\n" + "\n".join(r[1][-4000:] for r in failed))
        os.replace(lib_path + ".tmp", lib_path)
    finally:
        shutil.rmtree(objdir, ignore_errors=True)
    if verbose:
        print(log)
    return lib_path
