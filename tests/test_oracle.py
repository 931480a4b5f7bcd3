"""Pins the oracle (CPU only): the plain-C restatement oracle/nnc_port.c and the compiled reference oracle/_ref are
checked against the reference's literal known-answer vectors (tests/golden/literal_*.npz, typed from
test/unit/nnc/gemm.tests.c), against each other on seeded inputs, and against the committed CPU_REF fixtures."""
import hashlib
import json
import os

import numpy as np
import pytest

from ccv_b200 import nnc
from tests.util import assert_close, ref_exec, same, seeded

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def port():
    from oracle import port as p
    if not p.available():
        pytest.skip("oracle/_ref/libnnc_port.so not built (make -C oracle port)")
    return p


def test_port_matches_reference_literal_gemm_vectors(port):
    g = np.load(os.path.join(GOLDEN, "literal_gemm.npz"))
    assert np.array_equal(port.gemm_forw(g["a"], g["b"], None, 4, 3, 2, 0, 0), g["c"])
    assert np.array_equal(port.gemm_forw(g["a"], g["bt"], None, 4, 3, 2, 0, 1), g["c"])
    assert np.array_equal(port.gemm_forw(g["at"][0], g["bt"], None, 4, 3, 2, 1, 1), g["c"])
    assert np.array_equal(port.gemm_forw(g["a"], g["b"], g["bias"], 4, 3, 2, 0, 0), g["c_bias"])


@pytest.mark.ref
def test_compiled_reference_matches_its_own_literal_gemm_vectors(ref):
    g = np.load(os.path.join(GOLDEN, "literal_gemm.npz"))
    c = np.zeros((4, 3), np.float32)
    assert ref_exec(ref, nnc.CMD_GEMM_FORWARD(), None, 0, [g["a"], g["b"]], [c])[0] == 0
    assert np.array_equal(c, g["c"])
    assert ref_exec(ref, nnc.CMD_GEMM_FORWARD((0, 0), (0, 1)), None, 0, [g["a"], g["bt"], g["bias"]], [c])[0] == 0
    assert np.array_equal(c, g["c_bias"])


def test_port_matches_committed_cpu_ref_fixtures(port):
    g = np.load(os.path.join(GOLDEN, "cpuref_gemm.npz"))
    assert_close(port.gemm_forw(g["a"], g["w"], g["bias"], 12, 8, 20, 0, 1), g["b"], 1e-6, "gemm forward")
    h, dw, db = port.gemm_back(g["g"], g["a"], g["w"], 12, 8, 20, 0, 1)
    for a, n in ((h, "h"), (dw, "dw"), (db, "db")):
        assert_close(a, g[n], 1e-6, n)
    c = np.load(os.path.join(GOLDEN, "cpuref_conv.npz"))
    d = port.conv_desc(2, 9, 11, 8, 12, 3, 3, 2, 1)
    assert_close(port.conv_forw(d, c["x"], c["w"], c["bias"]), c["y"], 1e-6, "conv forward")
    gx, gw, gb = port.conv_back(d, c["gy"], c["x"], c["w"])
    assert_close(gx, c["gx"], 1e-6, "dgrad"), assert_close(gw, c["gw"], 1e-6, "wgrad"), assert_close(gb, c["gb"], 1e-6, "dbias")
    b = np.load(os.path.join(GOLDEN, "cpuref_bnorm.npz"))
    mean, var = b["mean0"].reshape(-1).copy(), b["var0"].reshape(-1).copy()
    y, sm, sis = port.bnorm_forw_train(b["x"], b["scale"].reshape(-1), b["bias"].reshape(-1), mean, var, 1e-4, 0.9)
    assert_close(y, b["y"], 1e-5, "bn y"), assert_close(mean, b["mean"].reshape(-1), 1e-6, "bn mean"), assert_close(var, b["var"].reshape(-1), 1e-5, "bn var")
    assert_close(sis, b["saved_inv_std"].reshape(-1), 1e-5, "bn inv std")
    f = np.load(os.path.join(GOLDEN, "cpuref_f2h.npz"))
    assert np.array_equal(port.float_to_half(f["f"]), f["h"])


@pytest.mark.ref
def test_port_matches_compiled_reference_on_seeded_inputs(port, ref):
    # GEMM NN with transposed a
    a, w = seeded((48, 33), 1, -1, 1), seeded((48, 21), 2, -1, 1)
    b = np.zeros((33, 21), np.float32)
    assert ref_exec(ref, nnc.CMD_GEMM_FORWARD((0, 1), (0, 0)), None, 0, [a, w], [b])[0] == 0
    assert_close(port.gemm_forw(a, w, None, 33, 21, 48, 1, 0), b, 1e-6, "gemm TN")
    # dilated convolution
    x, wt = seeded((1, 15, 15, 6), 3), seeded((10, 3, 3, 6), 4) / 54
    d = port.conv_desc(1, 15, 15, 6, 10, 3, 3, 1, 2, 2)
    y = np.zeros((1, 15, 15, 10), np.float32)
    hint = nnc.hint((1, 1), (2, 2))
    assert ref_exec(ref, nnc.CMD_CONVOLUTION_FORWARD(1, 10, 3, 3, 6, (2, 2)), hint, 0, [x, wt], [y])[0] == 0
    assert_close(port.conv_forw(d, x, wt, None), y, 1e-6, "dilated conv")
    # pooling (one image: CPU_REF ignores the rest of a batch)
    img = seeded((9, 9, 5), 5, -1, 1)
    for kind, fwd in (("max", nnc.CMD_MAX_POOL_FORWARD(3, 3)), ("avg", nnc.CMD_AVERAGE_POOL_FORWARD(3, 3))):
        out = np.zeros((5, 5, 5), np.float32)
        assert ref_exec(ref, fwd, nnc.hint((2, 2), (1, 1)), 0, [img], [out])[0] == 0
        p = port.pool_desc(1, 9, 9, 5, 3, 2, 1)
        got = (port.max_pool_forw if kind == "max" else port.avg_pool_forw)(p, img[None])[0]
        assert_close(got, out, 1e-6, kind + " pool")
    # softmax + sgd
    s = seeded((7, 100), 6, -3, 3)
    o = np.zeros_like(s)
    assert ref_exec(ref, nnc.CMD_SOFTMAX_FORWARD(), None, 0, [s], [o])[0] == 0
    assert_close(port.softmax_forw(s), o, 1e-6, "softmax")
    g, a2, m = seeded((5, 6), 7, -1, 1), seeded((5, 6), 8, -1, 1), seeded((5, 6), 9, -1, 1)
    bo, no = np.zeros_like(a2), np.zeros_like(a2)
    assert ref_exec(ref, nnc.CMD_SGD_FORWARD(0, 0.1, 0.5, 0.01, 0.9, 0.2), None, 0, [g, a2, m], [bo, no])[0] == 0
    pb, pn = port.sgd(g, a2, m, 0, 0.1, 0.5, 0.01, 0.9, 0.2)
    assert_close(pb, bo, 1e-6, "sgd b"), assert_close(pn, no, 1e-6, "sgd n")
    # half conversion: bit-exact against the reference's table method
    f = F2H_INPUT()
    if getattr(ref, "stored", False):  # the SHA-256 of the reference's bit patterns for these inputs (tests/golden/make_golden.py)
        want = json.load(open(os.path.join(GOLDEN, "reference_facts.json")))["float_to_half_sha256"]
        assert hashlib.sha256(np.ascontiguousarray(port.float_to_half(f), np.uint16).tobytes()).hexdigest() == want
    else:
        assert np.array_equal(port.float_to_half(f), ref.float_to_half(f))


def F2H_INPUT():
    return np.concatenate([seeded((20000,), 10, -70000, 70000), seeded((20000,), 11, -1e-4, 1e-4)]).astype(np.float32)


@pytest.mark.ref
def test_committed_fixtures_are_what_the_reference_produces(ref):
    """tests/golden/cpuref_*.npz must be reproducible from the compiled reference (guards against stale fixtures)."""
    g = np.load(os.path.join(GOLDEN, "cpuref_gemm.npz"))
    b = np.zeros_like(g["b"])
    assert ref_exec(ref, nnc.CMD_GEMM_FORWARD((0, 0), (0, 1)), None, 0, [g["a"], g["w"], g["bias"]], [b])[0] == 0
    assert np.array_equal(b, g["b"])


@pytest.mark.ref
def test_compiled_reference_reproduces_its_closed_form_convolution_cases(ref, port):
    """test/unit/nnc/forward.tests.c:14-44 ("convolutional network of 11x11 on 225x185 with uniform weights"): all-ones image and
    filters, stride 4 / border 1 from ccv_nnc_hint_auto -> 363 inside, 330 on the edges, 300 in the corners.  Checked on the
    compiled reference and on the plain-C restatement."""
    a, w, bias = np.ones((225, 185, 3), np.float32), np.ones((4, 11, 11, 3), np.float32), np.zeros((4,), np.float32)
    b = np.zeros((55, 45, 4), np.float32)
    cmd = nnc.CMD_CONVOLUTION_FORWARD(1, 4, 11, 11, 3)
    hint = nnc.hint((4, 4), (1, 1))  # what ccv_nnc_hint_auto derives for 225x185 -> 55x45 with an 11x11 window
    assert ref_exec(ref, cmd, hint, 0, [a, w, bias], [b])[0] == 0
    want = np.full((55, 45, 4), 363, np.float32)
    want[0, :], want[-1, :], want[:, 0], want[:, -1] = 330, 330, 330, 330
    want[0, 0], want[0, -1], want[-1, 0], want[-1, -1] = 300, 300, 300, 300
    assert same(b, want)
    d = port.conv_desc(1, 225, 185, 3, 4, 11, 11, 4, 1)
    assert np.array_equal(port.conv_forw(d, a[None], w, bias)[0], want)


@pytest.mark.ref
@pytest.mark.parametrize("causal", [0, 1])
def test_compiled_reference_attention_equals_the_composed_graph(ref, causal):
    """test/unit/nnc/attention.tests.c:14-97: SCALED_DOT_PRODUCT_ATTENTION_FORWARD on CPU_REF equals transpose -> scale -> q k^T ->
    softmax -> . v (here the composed side is float64 numpy; shapes scaled down from 32 x 128 x 8 x 64 / 96)."""
    B, S, H, D, Dv = 2, 32, 4, 16, 24
    q, k, v = seeded((B, S, H, D), 1), seeded((B, S, H, D), 2), seeded((B, S, H, Dv), 3)
    cmd = nnc._simple(nnc.CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_FORWARD)
    cmd.info.scaled_dot_product_attention.scale, cmd.info.scaled_dot_product_attention.is_causal = 1.0 / 8, causal
    o = np.zeros((B, S, H, Dv), np.float32)
    assert ref_exec(ref, cmd, None, 0, [q, k, v], [o, None])[0] == 0
    want = np.zeros_like(o, dtype=np.float64)
    for b in range(B):
        for h in range(H):
            s = (q[b, :, h].astype(np.float64) / 8) @ k[b, :, h].astype(np.float64).T
            if causal:
                s = np.where(np.arange(S)[None, :] <= np.arange(S)[:, None], s, -np.inf)
            e = np.exp(s - s.max(axis=1, keepdims=True))
            want[b, :, h] = (e / e.sum(axis=1, keepdims=True)) @ v[b, :, h].astype(np.float64)
    assert_close(o, want, 1e-5, "CPU_REF attention vs composed graph")


@pytest.mark.ref
def test_hint_auto_of_the_standalone_host_equals_the_reference():
    """ccv_nnc_hint_auto (lib/nnc/ccv_nnc_cmd.c:181-217) restated in ccv_b200/csrc/nnc_host.cu: stride and border (begin / end) for
    the window / input / output combinations the tests and the ResNet-50 driver use, byte for byte against the compiled reference."""
    import ctypes as C
    from ccv_b200 import abi
    from oracle import ref as r
    nnc.init()
    cases = HINT_AUTO_CASES
    stored = None if r.available() else json.load(open(os.path.join(GOLDEN, "reference_facts.json")))["hint_auto"]  # make_golden.py
    for i, case in enumerate(cases):
        size, a_dims, b_dims = case[:3]
        kind = case[3] if len(case) > 3 else "nhwc"
        fa = abi.CCV_TENSOR_FORMAT_NHWC if kind in ("nhwc", "mixed") else abi.CCV_TENSOR_FORMAT_NCHW
        fb = abi.CCV_TENSOR_FORMAT_NHWC if kind == "nhwc" else abi.CCV_TENSOR_FORMAT_NCHW
        info = abi.CmdParam()
        for j, d in enumerate(size):
            info.size.dim[j] = d
        pa = abi.tensor_param(abi.CCV_TENSOR_CPU_MEMORY, fa, abi.CCV_32F, list(a_dims), 0)
        pb = abi.tensor_param(abi.CCV_TENSOR_CPU_MEMORY, fb, abi.CCV_32F, list(b_dims), 0)
        mine, theirs = abi.Hint(), abi.Hint()
        nnc.lib().ccv_nnc_sm100_hint_auto(C.byref(info), C.byref(pa), C.byref(pb), C.byref(mine))
        if stored is None:
            r.ref().ref_hint_auto(C.byref(info), C.byref(pa), C.byref(pb), C.byref(theirs))
        else:
            C.memmove(C.byref(theirs), bytes.fromhex(stored[i]), C.sizeof(theirs))
        assert bytes(mine) == bytes(theirs), (size, a_dims, b_dims, list(mine.stride.dim[:3]), list(theirs.stride.dim[:3]), list(mine.border.begin[:3]), list(theirs.border.begin[:3]))


HINT_AUTO_CASES = [((11, 11, 3), (225, 185, 3), (55, 45, 4)), ((5, 3, 1), (17, 27, 1), (17, 27, 4)), ((3, 3, 3), (224, 224, 3), (112, 112, 32)),
    ((3, 3, 64), (56, 56, 64), (56, 56, 64)), ((3, 3, 128), (56, 56, 128), (28, 28, 128)), ((1, 1, 64), (56, 56, 64), (56, 56, 256)),
    ((2, 2, 256), (56, 56, 256), (28, 28, 256)), ((3, 3, 64), (112, 112, 64), (56, 56, 64)), ((7, 7, 2048), (7, 7, 2048), (1, 1, 2048)),
    ((3, 3, 8), (4, 13, 9, 8), (4, 7, 5, 16)),
    # windows smaller than the stride: the reference reports NEGATIVE borders (no clamping, ccv_nnc_cmd.c:212-214)
    ((1, 1, 16), (56, 56, 16), (28, 28, 16)), ((2, 2, 8), (60, 60, 8), (15, 15, 8)), ((1, 2, 4), (4, 33, 17, 4), (4, 11, 4, 4)),
    # NCHW, 3 and 4 dimensions; differing formats -> no hint
    ((3, 3, 8), (8, 32, 32), (8, 16, 16), "nchw"), ((5, 5, 8), (2, 8, 31, 29), (2, 8, 16, 15), "nchw"), ((3, 3, 8), (32, 32, 8), (8, 16, 16), "mixed")]


@pytest.mark.ref
@pytest.mark.parametrize("B,Sq,Sk,H,Hk,D,Dv,causal,masked", [(2, 24, 24, 4, 4, 16, 16, 0, 0), (1, 20, 28, 8, 2, 32, 24, 1, 0), (2, 16, 16, 2, 2, 8, 8, 0, 1)])
def test_port_attention_matches_compiled_reference(port, ref, B, Sq, Sk, H, Hk, D, Dv, causal, masked):
    """oracle/nnc_port.c:port_sdpa_forw (restated from ..._attention_cpu_ref.c:88-183) against CPU_REF itself: GQA, bottom-right
    causal alignment with Sq != Sk, additive mask."""
    q, k, v = seeded((B, Sq, H, D), 1, -1, 1), seeded((B, Sk, Hk, D), 2, -1, 1), seeded((B, Sk, Hk, Dv), 3, -1, 1)
    mask = np.where(np.random.RandomState(5).rand(Sq, Sk) < 0.3, -1e9, 0.0).astype(np.float32) if masked else None
    if masked:
        mask[np.arange(Sq), np.arange(Sq) % Sk] = 0
    cmd = nnc._simple(nnc.CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_FORWARD)
    cmd.info.scaled_dot_product_attention.scale, cmd.info.scaled_dot_product_attention.is_causal = 1.0 / np.sqrt(D), causal
    o = np.zeros((B, Sq, H, Dv), np.float32)
    ins = [q, k, v] + ([mask.reshape(1, 1, Sq, Sk)] if masked else [])
    assert ref_exec(ref, cmd, None, 0, ins, [o, None])[0] == 0
    assert_close(port.sdpa_forw(q, k, v, 1.0 / np.sqrt(D), causal, mask), o, 1e-6, "port attention")


@pytest.mark.ref
@pytest.mark.parametrize("rms", [0, 1])
def test_port_row_norms_match_compiled_reference(port, ref, rms):
    """oracle/nnc_port.c:port_row_norm_forw against CPU_REF's LAYER_NORM_FORWARD / RMSNORM_FORWARD over the last axis."""
    from ccv_b200 import abi
    shape, inner = (6, 10, 64), 64
    x, scale, bias = seeded(shape, 1, -1, 1), seeded((1, 1, inner), 2, 0.5, 1.5), seeded((1, 1, inner), 3, -1, 1)
    y, sm, sis = np.zeros(shape, np.float32), np.zeros((6, 10, 1), np.float32), np.zeros((6, 10, 1), np.float32)
    if rms:
        cmd = nnc._simple(abi.CCV_NNC_RMSNORM_FORWARD)
        cmd.info.rmsnorm.axis[0], cmd.info.rmsnorm.count, cmd.info.rmsnorm.epsilon = 2, 1, 1e-5
        assert ref_exec(ref, cmd, None, 0, [x, scale], [y, sis])[0] == 0
        yp, _, sp = port.row_norm_forw(x, scale, None, inner, 1e-5, rms=1)
    else:
        cmd = nnc._simple(abi.CCV_NNC_LAYER_NORM_FORWARD)
        cmd.info.lnorm.axis[0], cmd.info.lnorm.count, cmd.info.lnorm.epsilon, cmd.info.lnorm.elementwise_affine = 2, 1, 1e-5, 1
        assert ref_exec(ref, cmd, None, 0, [x, scale, bias], [y, sm, sis])[0] == 0
        yp, mp, sp = port.row_norm_forw(x, scale, bias, inner, 1e-5, rms=0)
        assert_close(mp.reshape(sm.shape), sm, 1e-6, "port mean")
    assert_close(yp, y, 1e-6, "port norm output"), assert_close(sp.reshape(sis.shape), sis, 1e-6, "port inv_std")
