"""Parity of the HBM-bound feeder commands (batch norm, relu, pooling, ewsum/add/mul, softmax, losses, SGD, set,
layout / datatype moves) against CCV_NNC_BACKEND_CPU_REF.  fp32 reductions: <= 1e-3 relative (north_star); the pure
elementwise ones are bit-exact or within 1e-6; index / datatype-conversion commands are bit-exact."""
import os

import numpy as np
import pytest

from ccv_b200 import abi
from tests.util import NCHW, NHWC, assert_close, gpu_exec, ref_exec, same, seeded

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
pytestmark = pytest.mark.gpu


@pytest.mark.ref
@pytest.mark.parametrize("shape", [(4, 7, 9, 32), (8, 14, 14, 64), (2, 5, 5, 20), (3, 6, 6, 7), (16, 1, 1, 2048)])
def test_batch_norm_forward_backward_vs_cpu_ref(gpu, ref, shape):
    """test/int/nnc/cudnn.tests.c:653-760 protocol (x in (0,1], seeded scale/bias), NHWC per-channel statistics."""
    nnc = gpu
    C = shape[-1]
    x = seeded(shape, 1, -1, 1)
    scale, bias = seeded((1, 1, 1, C), 2), seeded((1, 1, 1, C), 3)

    def fresh():
        return [seeded((1, 1, 1, C), 4), seeded((1, 1, 1, C), 5)]
    fwd = nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9)
    m_r, v_r = fresh()
    m_g, v_g = fresh()
    outs = lambda m, v: [np.zeros_like(x), m, v, np.zeros_like(m), np.zeros_like(m)]
    st_r, (y_r, m_r, v_r, sm_r, sis_r) = ref_exec(ref, fwd, None, 0, [x, scale, bias, m_r, v_r], outs(m_r, v_r))
    st_g, (y_g, m_g, v_g, sm_g, sis_g) = gpu_exec(nnc, fwd, None, 0, [x, scale, bias, m_g, v_g], outs(m_g, v_g))
    assert st_r == 0 and st_g == 0
    for a, b, n in ((y_g, y_r, "y"), (m_g, m_r, "running mean"), (v_g, v_r, "running var"), (sm_g, sm_r, "saved mean"), (sis_g, sis_r, "saved inv std")):
        assert_close(a, b, 1e-4, n)
    g = seeded(shape, 6, -1, 1)
    bwd = nnc.CMD_BATCH_NORM_BACKWARD(1e-4, 0, 0.9)
    ins = [g] + [None] * 4 + [x, scale] + [None] * 6 + [sm_r, sis_r]
    bouts = lambda: [np.zeros_like(x), np.zeros_like(scale), np.zeros_like(scale)]
    st_r, (h_r, ds_r, db_r) = ref_exec(ref, bwd, None, 0, ins, bouts())
    ins_g = [g] + [None] * 4 + [x, scale] + [None] * 6 + [sm_g, sis_g]  # each side's own saved statistics (compared above)
    st_g, (h_g, ds_g, db_g) = gpu_exec(nnc, bwd, None, 0, ins_g, bouts())
    assert st_r == 0 and st_g == 0
    assert_close(h_g, h_r, 1e-3, "dx")
    assert_close(ds_g, ds_r, 1e-3, "dscale")
    assert_close(db_g, db_r, 1e-3, "dbias")


@pytest.mark.ref
def test_batch_norm_inference_and_nchw(gpu, ref):
    nnc = gpu
    x = seeded((3, 6, 6, 24), 1, -1, 1)
    p = [seeded((1, 1, 1, 24), s) for s in (2, 3, 4, 5)]
    cmd = nnc.CMD_BATCH_NORM_FORWARD(1e-4, 1, 0.9)
    _, (y_r,) = ref_exec(ref, cmd, None, 0, [x] + p, [np.zeros_like(x)])
    st, (y_g,) = gpu_exec(nnc, cmd, None, 0, [x] + p, [np.zeros_like(x)])
    assert st == 0
    assert_close(y_g, y_r, 1e-5, "inference")
    xc = seeded((3, 10, 5, 7), 6, -1, 1)
    pc = [seeded((1, 10, 1, 1), s) for s in (7, 8)]
    m_r, v_r, m_g, v_g = (seeded((1, 10, 1, 1), s) for s in (9, 10, 9, 10))
    cmd = nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9, axes=(0, 2, 3))
    o = lambda m, v: [np.zeros_like(xc), m, v, np.zeros_like(m), np.zeros_like(m)]
    _, r = ref_exec(ref, cmd, None, 0, [xc] + pc + [m_r, v_r], o(m_r, v_r), fmt=NCHW)
    st, g = gpu_exec(nnc, cmd, None, 0, [xc] + pc + [m_g, v_g], o(m_g, v_g), fmt=NCHW)
    assert st == 0
    for a, b in zip(g, r):
        assert_close(a, b, 1e-4, "nchw")


def test_batch_norm_against_committed_cpu_ref_outputs(gpu):
    g = np.load(os.path.join(GOLDEN, "cpuref_bnorm.npz"))
    nnc = gpu
    m, v = g["mean0"].copy(), g["var0"].copy()
    st, outs = gpu_exec(nnc, nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9), None, 0, [g["x"], g["scale"], g["bias"], m, v], [np.zeros_like(g["x"]), m, v, np.zeros_like(m), np.zeros_like(m)])
    assert st == 0
    for a, n in zip(outs, ("y", "mean", "var", "saved_mean", "saved_inv_std")):
        assert_close(a, g[n], 1e-4, n)


@pytest.mark.ref
def test_relu_ewsum_add_mul_scalar_mul_vs_cpu_ref(gpu, ref):
    nnc = gpu
    a, b, c = seeded((4, 9, 9, 33), 1, -1, 1), seeded((4, 9, 9, 33), 2, -1, 1), seeded((4, 9, 9, 33), 3, -1, 1)
    zeros = lambda: [np.zeros_like(a)]
    for cmd, ins in ((nnc.CMD_RELU_FORWARD(), [a]), (nnc.CMD_EWSUM_FORWARD(), [a, b, c]), (nnc.CMD_ADD_FORWARD(0.5, -1.25), [a, b]), (nnc.CMD_MUL_FORWARD(0.7), [a, b]), (nnc.CMD_SCALAR_MUL_FORWARD(-2.5), [a])):
        _, (r,) = ref_exec(ref, cmd, None, 0, ins, zeros())
        st, (g,) = gpu_exec(nnc, cmd, None, 0, ins, zeros())
        assert st == 0
        assert_close(g, r, 1e-6, hex(cmd.cmd))
    # relu backward uses the forward OUTPUT as the mask (relu/ccv_nnc_relu_cpu_ref.c:51)
    y = np.maximum(a, 0)
    _, (r,) = ref_exec(ref, nnc.CMD_RELU_BACKWARD(), None, 0, [b, None, y], zeros())
    st, (g,) = gpu_exec(nnc, nnc.CMD_RELU_BACKWARD(), None, 0, [b, None, y], zeros())
    assert st == 0 and same(g, r)
    # broadcast add: bias-like [33] into [4,9,9,33], and its gradient (a reduction)
    bias = seeded((33,), 4)
    _, (r,) = ref_exec(ref, nnc.CMD_ADD_FORWARD(1, 1), None, 0, [a, bias], zeros())
    st, (g,) = gpu_exec(nnc, nnc.CMD_ADD_FORWARD(1, 1), None, 0, [a, bias], zeros())
    assert st == 0
    assert_close(g, r, 1e-6, "broadcast add")
    _, (ha_r, hb_r) = ref_exec(ref, nnc.CMD_ADD_BACKWARD(1, 1), None, 0, [c, a, bias], [np.zeros_like(a), np.zeros_like(bias)])
    st, (ha_g, hb_g) = gpu_exec(nnc, nnc.CMD_ADD_BACKWARD(1, 1), None, 0, [c, a, bias], [np.zeros_like(a), np.zeros_like(bias)])
    assert st == 0
    assert_close(ha_g, ha_r, 1e-6, "add back a")
    assert_close(hb_g, hb_r, 1e-4, "add back bias")


@pytest.mark.ref
@pytest.mark.parametrize("kind,H,W,C,R,st,pad", [("max", 13, 13, 8, 3, 2, 1), ("max", 12, 10, 5, 2, 2, 0), ("avg", 14, 14, 16, 2, 2, 0), ("avg", 7, 7, 32, 7, 1, 0), ("avg", 9, 9, 6, 3, 1, 1)])
def test_pooling_forward_backward_vs_cpu_ref(gpu, ref, kind, H, W, C, R, st, pad):
    """CPU_REF pools only walk image 0 of a batch (SURVEY.md 0.6), so the oracle is called once per image."""
    nnc = gpu
    N = 3
    P, Q = (H + 2 * pad - R) // st + 1, (W + 2 * pad - R) // st + 1
    a = seeded((N, H, W, C), 1, -1, 1)
    a = np.round(a * 8) / 8 if kind == "max" else a  # ties exercise the "every maximum gets the gradient" rule
    hint = nnc.hint((st, st), (pad, pad))
    fwd = (nnc.CMD_MAX_POOL_FORWARD if kind == "max" else nnc.CMD_AVERAGE_POOL_FORWARD)(R, R)
    bwd = (nnc.CMD_MAX_POOL_BACKWARD if kind == "max" else nnc.CMD_AVERAGE_POOL_BACKWARD)(R, R)
    b_r = [np.zeros((P, Q, C), np.float32) for _ in range(N)]
    for n in range(N):
        assert ref_exec(ref, fwd, hint, 0, [np.ascontiguousarray(a[n])], [b_r[n]])[0] == 0
    stt, (b_g,) = gpu_exec(nnc, fwd, hint, 0, [a], [np.zeros((N, P, Q, C), np.float32)])
    assert stt == 0
    for n in range(N):  # normalised per image: no looser than over the batch
        assert_close(b_g[n], b_r[n], 1e-6, "forward")
    g = seeded((N, P, Q, C), 2, -1, 1)
    h_r = [np.zeros((H, W, C), np.float32) for _ in range(N)]
    for n in range(N):
        ins = [np.ascontiguousarray(g[n]), np.ascontiguousarray(a[n]), b_r[n]]
        assert ref_exec(ref, bwd, hint, 0, ins, [h_r[n]])[0] == 0
    stt, (h_g,) = gpu_exec(nnc, bwd, hint, 0, [g, a, b_g], [np.zeros_like(a)])  # its own forward output (compared above)
    assert stt == 0
    for n in range(N):
        assert_close(h_g[n], h_r[n], 1e-5, "backward")


@pytest.mark.ref
def test_softmax_and_losses_vs_cpu_ref(gpu, ref):
    nnc = gpu
    a = seeded((37, 1000), 1, -4, 4)
    _, (p_r,) = ref_exec(ref, nnc.CMD_SOFTMAX_FORWARD(), None, 0, [a], [np.zeros_like(a)])
    st, (p_g,) = gpu_exec(nnc, nnc.CMD_SOFTMAX_FORWARD(), None, 0, [a], [np.zeros_like(a)])
    assert st == 0
    assert_close(p_g, p_r, 1e-5, "softmax")
    g = seeded(a.shape, 2, -1, 1)
    _, (h_r,) = ref_exec(ref, nnc.CMD_SOFTMAX_BACKWARD(), None, 0, [g, None, p_r], [np.zeros_like(a)])
    st, (h_g,) = gpu_exec(nnc, nnc.CMD_SOFTMAX_BACKWARD(), None, 0, [g, None, p_g], [np.zeros_like(a)])  # each side's own probabilities
    assert st == 0
    assert_close(h_g, h_r, 1e-4, "softmax backward")
    labels_f = np.random.RandomState(3).randint(0, 1000, size=(37,)).astype(np.float32)
    labels_i = labels_f.astype(np.int32)
    onehot = np.zeros_like(a)
    onehot[np.arange(37), labels_i] = 1
    gl = seeded((37,), 4)
    for lab in (labels_f, labels_i, onehot):
        for trims in ((0.0, 1.0), (0.1 / 999, 0.9)):
            if lab is onehot and trims != (0.0, 1.0):
                continue
            fwd, bwd = nnc.CMD_CATEGORICAL_CROSSENTROPY_FORWARD(*trims), nnc.CMD_CATEGORICAL_CROSSENTROPY_BACKWARD(*trims)
            _, (c_r,) = ref_exec(ref, fwd, None, 0, [p_r, lab], [np.zeros((37,), np.float32)])
            st, (c_g,) = gpu_exec(nnc, fwd, None, 0, [p_g, lab], [np.zeros((37,), np.float32)])
            assert st == 0
            assert_close(c_g, c_r, 1e-5, "cce forward")
            _, (h_r,) = ref_exec(ref, bwd, None, 0, [gl, p_r, lab], [np.zeros_like(a)])
            st, (h_g,) = gpu_exec(nnc, bwd, None, 0, [gl, p_g, lab], [np.zeros_like(a)])
            assert st == 0
            assert_close(h_g, h_r, 1e-5, "cce backward")
            sf, sb = nnc.CMD_SOFTMAX_CROSSENTROPY_FORWARD(*trims), nnc.CMD_SOFTMAX_CROSSENTROPY_BACKWARD(*trims)
            _, (c_r, d_r) = ref_exec(ref, sf, None, 0, [a, lab], [np.zeros((37,), np.float32), np.zeros_like(a)])
            st, (c_g, d_g) = gpu_exec(nnc, sf, None, 0, [a, lab], [np.zeros((37,), np.float32), np.zeros_like(a)])
            assert st == 0
            assert_close(c_g, c_r, 1e-5, "softmax-ce loss")
            assert_close(d_g, d_r, 1e-5, "softmax-ce probabilities")
            _, (h_r,) = ref_exec(ref, sb, None, 0, [gl, None, None, lab, None, d_r], [np.zeros_like(a)])
            st, (h_g,) = gpu_exec(nnc, sb, None, 0, [gl, None, None, lab, None, d_g], [np.zeros_like(a)])  # each side's own probabilities
            assert st == 0
            assert_close(h_g, h_r, 1e-5, "softmax-ce backward")


@pytest.mark.ref
@pytest.mark.parametrize("nesterov", [0, 1])
def test_sgd_vs_cpu_ref(gpu, ref, nesterov):
    """test/int/nnc/sgd.tests.c protocol."""
    nnc = gpu
    g, a, m = seeded((10, 7, 5, 3), 1, -1, 1), seeded((10, 7, 5, 3), 2, -1, 1), seeded((10, 7, 5, 3), 3, -1, 1)
    cmd = nnc.CMD_SGD_FORWARD(nesterov, 0.01, 1.0 / 128, 0.0005, 0.9, 0.0 if nesterov else 0.1)
    _, (b_r, n_r) = ref_exec(ref, cmd, None, 0, [g, a, m], [np.zeros_like(a), np.zeros_like(a)])
    st, (b_g, n_g) = gpu_exec(nnc, cmd, None, 0, [g, a, m], [np.zeros_like(a), np.zeros_like(a)])
    assert st == 0
    assert_close(b_g, b_r, 1e-6, "sgd b")
    assert_close(n_g, n_r, 1e-6, "sgd momentum")


def test_datatype_conversion_is_bit_exact_with_the_reference_tables(gpu):
    """f32 -> f16 must TRUNCATE like lib/ccv_util.c:1434-1440 (SURVEY.md 0.7); fixture made by the reference itself."""
    g = np.load(os.path.join(GOLDEN, "cpuref_f2h.npz"))
    nnc = gpu
    f, want = g["f"], g["h"]
    tf = nnc.gpu_tensor([f.size], datatype=abi.CCV_32F); tf.upload(f)
    th = nnc.gpu_tensor([f.size], datatype=abi.CCV_16F)
    assert nnc.cmd_exec(nnc.CMD_DATATYPE_CONVERSION_FORWARD(), None, 0, [tf], [th]) == 0
    got = th.download().view(np.uint16)
    assert np.array_equal(got, want), "first mismatch at %d" % int(np.argmax(got != want))
    # and back: half -> float is exact
    tb = nnc.gpu_tensor([f.size], datatype=abi.CCV_32F)
    assert nnc.cmd_exec(nnc.CMD_DATATYPE_CONVERSION_FORWARD(), None, 0, [th], [tb]) == 0
    back = tb.download()
    finite = np.isfinite(back)
    assert np.array_equal(back[finite], want.view(np.float16).astype(np.float32)[finite])
    for t in (tf, th, tb):
        t.free()


@pytest.mark.ref
def test_set_transfer_format_transform_transpose_are_bit_exact(gpu, ref):
    nnc = gpu
    a = seeded((2, 5, 6, 7), 1, -1, 1)
    st, (s,) = gpu_exec(nnc, nnc.CMD_SET_FORWARD(1.5), None, 0, [], [np.zeros_like(a)])
    assert st == 0 and np.all(s == 1.5)
    st, (c,) = gpu_exec(nnc, nnc.CMD_DATA_TRANSFER_FORWARD(), None, 0, [a], [np.zeros_like(a)])
    assert st == 0 and np.array_equal(c, a)
    # NHWC [2,5,6,7] -> NCHW [2,7,5,6]
    out_r, out_g = np.zeros((2, 7, 5, 6), np.float32), np.zeros((2, 7, 5, 6), np.float32)
    ref_exec(ref, nnc.CMD_FORMAT_TRANSFORM_FORWARD(), None, 0, [a], [out_r], in_fmts=[NHWC], out_fmts=[NCHW])
    st, (out_g,) = gpu_exec(nnc, nnc.CMD_FORMAT_TRANSFORM_FORWARD(), None, 0, [a], [out_g], in_fmts=[NHWC], out_fmts=[NCHW])
    assert st == 0 and same(out_g, out_r) and np.array_equal(out_g, a.transpose(0, 3, 1, 2))
    t_r, t_g = np.zeros((2, 6, 5, 7), np.float32), np.zeros((2, 6, 5, 7), np.float32)
    ref_exec(ref, nnc.CMD_TRANSPOSE_FORWARD(1, 2), None, 0, [a], [t_r])
    st, (t_g,) = gpu_exec(nnc, nnc.CMD_TRANSPOSE_FORWARD(1, 2), None, 0, [a], [t_g])
    assert st == 0 and same(t_g, t_r)


@pytest.mark.ref
@pytest.mark.parametrize("N,H,C,K,R,relu,offset", [(8, 28, 64, 128, 3, 1, 0.0), (16, 14, 256, 64, 1, 0, 0.0), (4, 32, 3, 32, 3, 1, 0.0),
                                                     (32, 28, 64, 128, 3, 0, 60.0),   # 196 output tiles (some CTAs own two), channel mean / std ~ 100
                                                     (8, 14, 128, 512, 1, 1, -80.0),  # two column blocks of 256
                                                     (4, 7, 64, 2048, 1, 0, 25.0)])   # eight column blocks: a CTA's tiles alternate between two of them
def test_convolution_epilogue_statistics_feed_the_batch_norm(gpu, ref, N, H, C, K, R, relu, offset):
    """Graph rewrite (f) of ccv_nnc_sm100_graph_fuse: CONVOLUTION_FORWARD -> BATCH_NORM_FORWARD(train) [-> RELU in place].  The
    convolution's tensor-core epilogue folds its output into per-(CTA, warp quarter) shifted sums and the batch norm skips its
    statistics pass.  Checked against CPU_REF running the same three commands one by one (two-pass variance,
    norm/ccv_nnc_batch_norm_cpu_ref.c:66-110): y within the TF32 bound, saved mean / inv_std / running statistics within 1e-3,
    also when a convolution bias puts the channel means ~100 standard deviations from zero (the case in which an unshifted
    E[y^2] - E[y]^2 loses the variance), and the result is bit-identical from run to run (no atomics)."""
    nnc = gpu
    pad = R // 2
    x, w, b = seeded((N, H, H, C), 1, -1, 1), seeded((K, R, R, C), 2, -1, 1) / (R * R * C) ** 0.5, seeded((K,), 3, -1, 1) + np.float32(offset)
    scale, bias = seeded((1, 1, 1, K), 4, 0.5, 1.5), seeded((1, 1, 1, K), 5, -1, 1)
    hint = nnc.hint((1, 1), (pad, pad))
    conv = nnc.CMD_CONVOLUTION_FORWARD(1, K, R, R, C)
    bn = nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9)
    # oracle: conv, bn, relu one by one
    y = np.zeros((N, H, H, K), np.float32)
    assert ref_exec(ref, conv, hint, 0, [x, w, b], [y])[0] == 0
    mean, var = np.zeros((1, 1, 1, K), np.float32), np.ones((1, 1, 1, K), np.float32)
    z, sm, sis = np.zeros_like(y), np.zeros((1, 1, 1, K), np.float32), np.zeros((1, 1, 1, K), np.float32)
    assert ref_exec(ref, bn, None, 0, [y, scale, bias, mean, var], [z, mean, var, sm, sis])[0] == 0
    if relu:
        np.maximum(z, 0, out=z)
    # GPU: the same commands as a graph, fused
    stream = nnc.Stream(0)
    T = lambda a: nnc.gpu_tensor(list(a.shape)).upload(a)
    tx, tw, tb, tscale, tbias = T(x), T(w), T(b), T(scale), T(bias)
    tmean, tvar = T(np.zeros((1, 1, 1, K), np.float32)), T(np.ones((1, 1, 1, K), np.float32))
    ty, tz, tsm, tsis = (nnc.gpu_tensor(s) for s in ([N, H, H, K], [N, H, H, K], [1, 1, 1, K], [1, 1, 1, K]))
    g = nnc.Graph()
    g.exec_new(conv, hint, 0, [tx, tw, tb], [ty])
    g.exec_new(bn, None, 0, [ty, tscale, tbias, tmean, tvar], [tz, tmean, tvar, tsm, tsis])
    if relu:
        g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [tz], [tz])
    g.fuse()
    kinds = [k for _, k, _, _ in g.nodes()]
    assert kinds == ([6, 1] if relu else [6, 7]), kinds
    assert g.run(stream) == 0
    stream.wait()
    assert_close(ty.download(), y, 1e-3, "convolution output")
    assert_close(tsm.download(), sm, 1e-3, "saved mean"), assert_close(tsis.download(), sis, 1e-3, "saved inv_std")
    assert_close(tmean.download(), mean, 1e-3, "running mean"), assert_close(tvar.download(), var, 1e-3, "running var")
    assert_close(tz.download(), z, 2e-3, "normalised output")
    # deterministic: a second run of the same graph reproduces every bit of the statistics and of the output
    first = [t.download() for t in (tsm, tsis, tz)]
    tmean.upload(np.zeros((1, 1, 1, K), np.float32)), tvar.upload(np.ones((1, 1, 1, K), np.float32))
    assert g.run(stream) == 0
    stream.wait()
    for t, f in zip((tsm, tsis, tz), first):
        assert np.array_equal(t.download(), f)
    for t in (tx, tw, tb, tscale, tbias, tmean, tvar, ty, tz, tsm, tsis, g, stream):
        t.free()


@pytest.mark.parametrize("C,relu", [(64, 0), (256, 1), (2048, 0)])
def test_batch_norm_backward_also_writes_the_convolution_bias_gradient(gpu, C, relu):
    """Graph rewrite (g): [RELU_BACKWARD ;] BATCH_NORM_BACKWARD ; CONVOLUTION_BACKWARD(g = the batch norm's dx).  The fused list must
    give the convolution the same dbias = sum over pixels of dx (mathematically 0 behind a batch norm, so the comparison is
    against the magnitude of the summands), the same dx and the same filter gradient as the unfused list."""
    nnc = gpu
    N, H, Cin, R = 8, 7, 32, 1
    stream = nnc.Stream(0)
    rs = np.random.RandomState(3)
    x_in, w = seeded((N, H, H, Cin), 1, -1, 1), seeded((C, R, R, Cin), 2, -1, 1) / Cin ** 0.5
    y = rs.randn(N, H, H, C).astype(np.float32)            # the convolution's output = the batch norm's input
    gy = rs.randn(N, H, H, C).astype(np.float32)
    scale, bias = seeded((1, 1, 1, C), 4, 0.5, 1.5), seeded((1, 1, 1, C), 5, -1, 1)
    mean = y.mean(axis=(0, 1, 2)).reshape(1, 1, 1, C).astype(np.float32)
    inv_std = (1.0 / np.sqrt(y.var(axis=(0, 1, 2)) + 1e-4)).reshape(1, 1, 1, C).astype(np.float32)
    z = np.maximum((y - mean) * inv_std * scale + bias, 0).astype(np.float32)  # relu(bn(y)), the mask source

    def run(fuse):
        T = lambda a: nnc.gpu_tensor(list(a.shape)).upload(a)
        t = dict(x=T(x_in), w=T(w), y=T(y), g=T(gy), scale=T(scale), bias=T(bias), mean=T(mean), istd=T(inv_std), z=T(z))
        t.update(dx=nnc.gpu_tensor([N, H, H, C]), dscale=nnc.gpu_tensor([1, 1, 1, C]), dbias=nnc.gpu_tensor([1, 1, 1, C]),
                 h=nnc.gpu_tensor([N, H, H, Cin]), dw=nnc.gpu_tensor([C, R, R, Cin]), cdb=nnc.gpu_tensor([C]), mv=T(np.zeros((1, 1, 1, C), np.float32)))
        gr = nnc.Graph()
        # a forward batch norm node so that the ReLU-backward fusion can find the bias of the masked activation
        gr.exec_new(nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9), None, 0, [t["y"], t["scale"], t["bias"], t["mv"], t["mv"]], [t["z"], t["mv"], t["mv"], t["mean"], t["istd"]])
        if relu:
            gr.exec_new(nnc.CMD_RELU_BACKWARD(), None, 0, [t["g"], None, t["z"]], [t["g"]])
        bn_in = [t["g"]] + [None] * 4 + [t["y"], t["scale"]] + [None] * 6 + [t["mean"], t["istd"]]
        gr.exec_new(nnc.CMD_BATCH_NORM_BACKWARD(1e-4, 0, 0.9), None, 0, bn_in, [t["dx"], t["dscale"], t["dbias"]])
        gr.exec_new(nnc.CMD_CONVOLUTION_BACKWARD(1, C, R, R, Cin), nnc.hint((1, 1), (0, 0)), 0, [t["dx"], t["x"], t["w"]], [t["h"], t["dw"], t["cdb"]])
        if fuse:
            gr.fuse()
            kinds = [k for _, k, _, _ in gr.nodes()]
            assert (2 in kinds) if relu else (8 in kinds), kinds
        assert gr.run(stream) == 0
        stream.wait()
        res = {k: t[k].download() for k in ("dx", "dw", "cdb", "h", "dscale", "dbias")}
        for v in t.values():
            v.free()
        gr.free()
        return res

    a, b = run(False), run(True)
    for k in ("dx", "dw", "h", "dscale", "dbias"):
        assert_close(b[k], a[k], 1e-5, k)
    bound = 1e-5 * np.abs(a["dx"]).reshape(-1, C).sum(axis=0).max()
    assert np.abs(b["cdb"] - a["cdb"]).max() <= bound, (np.abs(b["cdb"] - a["cdb"]).max(), bound)
    stream.free()
