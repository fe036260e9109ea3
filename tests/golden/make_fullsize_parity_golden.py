"""Generates tests/golden/sepconv_fullsize_ref.npz: SHA-256 digests of the inputs of tests/test_gpu_fullsize_parity.py and
of the reference kernel's forward, grad_vertical and grad_horizontal on them, so that the full-size parity test runs
without a build of the reference.  The inputs are made on the GPU by the test's own seeded generators:

    python tests/golden/make_fullsize_parity_golden.py OUT.npz          (on a B200)

then copy OUT.npz to tests/golden/sepconv_fullsize_ref.npz.  The reference's outputs are computed by the CPU oracle's
reference-order restatement (oracle/sepconv_oracle.c), which is bit-equal to libs/sepconv/src/SeparableConvolution_kernel.cu
compiled verbatim for sm_100a (tests/golden/sepconv_ref.npz); when oracle/_ref is built, every output is also checked
against that build here."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
import oracle  # noqa: E402
from tests import _ref_cuda  # noqa: E402
from tests.test_gpu_fullsize_parity import CASES, case_inputs, sha256, tail_inputs  # noqa: E402


def _forward(inp, v, h):
    out = torch.from_numpy(oracle.sepconv_forward_reforder(*(t.cpu().numpy() for t in (inp, v, h))))
    if _ref_cuda.available():
        assert torch.equal(out, _ref_cuda.forward(inp, v, h).cpu())
    return out


def main(dst):
    dev = torch.device("cuda")
    out = {}
    for name in CASES:
        inp, v, h, g = case_inputs(name, dev)
        ni, nv, nh, ng = (t.cpu().numpy() for t in (inp, v, h, g))
        gv = torch.from_numpy(oracle.sepconv_grad_vertical_reforder(ng, ni, nh))
        gh = torch.from_numpy(oracle.sepconv_grad_horizontal_reforder(ng, ni, nv))
        if _ref_cuda.available():
            _, ref_gv, ref_gh = _ref_cuda.backward(g, inp, v, h)
            assert torch.equal(gv, ref_gv.cpu()) and torch.equal(gh, ref_gh.cpu())
        out[name + "_inputs_sha256"] = sha256(inp, v, h, g)
        out[name + "_out_sha256"] = sha256(_forward(inp, v, h))
        out[name + "_gv_sha256"] = sha256(gv)
        out[name + "_gh_sha256"] = sha256(gh)
        del inp, v, h, g, gv, gh
        torch.cuda.empty_cache()
        print(name, flush=True)
    inp, inp2, taps = tail_inputs(dev)
    out["tail_512_inputs_sha256"] = sha256(inp, inp2, *taps)
    out["tail_512_ref1_sha256"] = sha256(_forward(inp, taps[0], taps[1]))
    out["tail_512_ref2_sha256"] = sha256(_forward(inp2, taps[2], taps[3]))
    np.savez_compressed(dst, **out)
    print("wrote", dst, sorted(out))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "sepconv_fullsize_ref.npz"))
