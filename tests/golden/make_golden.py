"""Regenerates tests/golden/*.npz from the reference's own known-answer tests and from the compiled reference
(oracle/_ref/libccv_ref.so).  Run where the reference sources are present and `make -C oracle` has built the compiled reference:

    python tests/golden/make_golden.py          # everything below
    python tests/golden/make_golden.py facts    # reference_facts.json only

The CPU_REF outputs of the parity tests (tests/golden/cpu_ref/) are written by the tests themselves: run the suite on a GPU
machine with CCV_REF_RECORD=1 and the compiled reference present (tests/util.py).

Three kinds of fixtures here:
  literal_*   inputs + expected outputs typed from the reference's unit tests (test/unit/nnc/gemm.tests.c etc.); these
              pin the oracle itself.
  cpuref_*    seeded inputs + the outputs CCV_NNC_BACKEND_CPU_REF produced for them here; these travel to the GPU box
              so parity can be checked even without the compiled reference.
  reference_facts.json   the reference's struct layouts, ccv_nnc_hint_auto results and the digest of its float -> half bit patterns
                         (tests/test_abi.py, tests/test_oracle.py).
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from ccv_b200 import nnc  # noqa: E402
from oracle import ref  # noqa: E402
from tests.util import seeded  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def literal_gemm():
    """test/unit/nnc/gemm.tests.c:13-200 (forward cases, hand-computed expectations)."""
    a = np.array([[1, 2], [3, 4], [5, 6], [7, 8]], np.float32)
    b = np.array([[7, 8, 9], [10, 11, 12]], np.float32)
    c = a.astype(np.float64) @ b.astype(np.float64)
    bias = np.array([22, 23, 24], np.float32)
    return dict(a=a, b=b, c=c.astype(np.float32), bt=np.ascontiguousarray(b.T), at=np.ascontiguousarray(a.T)[None], bias=bias,
                c_bias=(c + bias).astype(np.float32))


def cpuref_cases():
    cases = {}
    # GEMM forward NT with bias (dense layer form) and backward
    a, w, bias = seeded((12, 20), 1, -1, 1), seeded((8, 20), 2, -1, 1), seeded((8,), 3)
    b = np.zeros((12, 8), np.float32)
    assert ref.run(nnc.CMD_GEMM_FORWARD((0, 0), (0, 1)), None, 0, [a, w, bias], [b]) == 0
    g = seeded((12, 8), 4, -1, 1)
    h, dw, db = np.zeros_like(a), np.zeros_like(w), np.zeros_like(bias)
    assert ref.run(nnc.CMD_GEMM_BACKWARD((0, 0), (0, 1)), None, 0, [g, a, w], [h, dw, db]) == 0
    cases["gemm"] = dict(a=a, w=w, bias=bias, b=b, g=g, h=h, dw=dw, db=db)
    # convolution 3x3 stride 2 pad 1 with bias, forward + backward (NHWC)
    x, wt, cb = seeded((2, 9, 11, 8), 5), seeded((12, 3, 3, 8), 6) / 72, seeded((12,), 7)
    y = np.zeros((2, 5, 6, 12), np.float32)
    hint = nnc.hint((2, 2), (1, 1))
    assert ref.run(nnc.CMD_CONVOLUTION_FORWARD(1, 12, 3, 3, 8), hint, 0, [x, wt, cb], [y]) == 0
    gy = seeded(y.shape, 8)
    gx, gw, gb = np.zeros_like(x), np.zeros_like(wt), np.zeros_like(cb)
    assert ref.run(nnc.CMD_CONVOLUTION_BACKWARD(1, 12, 3, 3, 8), hint, 0, [gy, x, wt], [gx, gw, gb]) == 0
    cases["conv"] = dict(x=x, w=wt, bias=cb, y=y, gy=gy, gx=gx, gw=gw, gb=gb)
    # batch norm training forward
    bx = seeded((4, 5, 6, 16), 9, -1, 1)
    scale, bb = seeded((1, 1, 1, 16), 10), seeded((1, 1, 1, 16), 11)
    mean, var = seeded((1, 1, 1, 16), 12), seeded((1, 1, 1, 16), 13)
    mean0, var0 = mean.copy(), var.copy()
    by, sm, sis = np.zeros_like(bx), np.zeros_like(mean), np.zeros_like(mean)
    assert ref.run(nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9), None, 0, [bx, scale, bb, mean, var], [by, mean, var, sm, sis]) == 0
    cases["bnorm"] = dict(x=bx, scale=scale, bias=bb, mean0=mean0, var0=var0, y=by, mean=mean, var=var, saved_mean=sm, saved_inv_std=sis)
    # float -> half conversion bit patterns (truncating, lib/ccv_util.c:1434-1440)
    f = np.concatenate([seeded((4096,), 14, -70000, 70000), seeded((4096,), 15, -1e-4, 1e-4), np.array([0.0, -0.0, 65504.0, 65520.0, 1e-8, 6.1e-5, 5.9e-8, np.inf, -np.inf], np.float32)]).astype(np.float32)
    cases["f2h"] = dict(f=f, h=ref.float_to_half(f))
    return cases


def reference_facts():
    """What the compiled reference reports about itself: its struct sizes / field offsets (ref_shim.c:ref_abi_sizes) and the hints
    ccv_nnc_hint_auto derives for tests/test_oracle.py HINT_AUTO_CASES (raw ccv_nnc_hint_t bytes, hex)."""
    import ctypes as C
    from ccv_b200 import abi
    from tests.test_oracle import HINT_AUTO_CASES
    sizes = (C.c_int * 10)()
    ref.ref().ref_abi_sizes(sizes)
    hints = []
    for case in HINT_AUTO_CASES:
        size, a_dims, b_dims = case[:3]
        kind = case[3] if len(case) > 3 else "nhwc"
        fa = abi.CCV_TENSOR_FORMAT_NHWC if kind in ("nhwc", "mixed") else abi.CCV_TENSOR_FORMAT_NCHW
        fb = abi.CCV_TENSOR_FORMAT_NHWC if kind == "nhwc" else abi.CCV_TENSOR_FORMAT_NCHW
        info = abi.CmdParam()
        for j, d in enumerate(size):
            info.size.dim[j] = d
        pa = abi.tensor_param(abi.CCV_TENSOR_CPU_MEMORY, fa, abi.CCV_32F, list(a_dims), 0)
        pb = abi.tensor_param(abi.CCV_TENSOR_CPU_MEMORY, fb, abi.CCV_32F, list(b_dims), 0)
        h = abi.Hint()
        ref.ref().ref_hint_auto(C.byref(info), C.byref(pa), C.byref(pb), C.byref(h))
        hints.append(bytes(h).hex())
    from tests.test_oracle import F2H_INPUT
    return dict(abi_sizes=list(sizes), hint_auto=hints, float_to_half_sha256=hashlib.sha256(ref.float_to_half(F2H_INPUT()).tobytes()).hexdigest())


if __name__ == "__main__":
    if sys.argv[1:] == ["facts"]:  # only reference_facts.json
        json.dump(reference_facts(), open(os.path.join(OUT, "reference_facts.json"), "w"), indent=1)
        sys.exit(0)
    np.savez(os.path.join(OUT, "literal_gemm.npz"), **literal_gemm())
    for name, d in cpuref_cases().items():
        np.savez(os.path.join(OUT, "cpuref_%s.npz" % name), **d)
    json.dump(reference_facts(), open(os.path.join(OUT, "reference_facts.json"), "w"), indent=1)
    print("wrote", sorted(os.listdir(OUT)))
