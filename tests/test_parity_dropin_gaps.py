"""Behaviours the reference's own GPU test programs exercise (test/int/nnc/cudnn.tests.c, cublas.tests.c, sgd.tests.c, schedule.tests.c)
that the first drop-in run (integration/, SURVEY.md 8f-1) showed missing, now as parity tests of the backend itself:
broadcasting MUL backward, GEMM with two batch axes and views, SET for every datatype, int32 EWSUM, 16-bit tensors on the
fp32-only commands (softmax, add, mul, scalar mul, softmax cross-entropy), NCHW pooling, SGD with 16-bit parameters."""
import numpy as np
import pytest

from ccv_b200 import abi
from tests.util import NCHW, NHWC, assert_close, gpu_exec, gpu_exec16, max_abs_diff, ref_exec, round16, same, seeded

pytestmark = [pytest.mark.gpu, pytest.mark.ref]


@pytest.mark.parametrize("with_g", [True, False])
def test_mul_backward_broadcast(gpu, ref, with_g):
    """test/int/nnc/cudnn.tests.c:5169-5336: a [4, 1] * b [2] -> c [4, 2]; each gradient sums over the axes its operand was broadcast along"""
    nnc = gpu
    a, b, g = seeded((4, 1), 1, -1, 1), seeded((2,), 2, -1, 1), seeded((4, 2), 3, -1, 1)
    ins = [g if with_g else None, a, b]
    cmd = nnc.CMD_MUL_BACKWARD(0.5)
    _, (da_r, db_r) = ref_exec(ref, cmd, None, 0, ins, [np.zeros_like(a), np.zeros_like(b)])
    st, (da_g, db_g) = gpu_exec(nnc, cmd, None, 0, ins, [np.zeros_like(a), np.zeros_like(b)])
    assert st == 0
    assert_close(da_g, da_r, 1e-6, "da"), assert_close(db_g, db_r, 1e-6, "db")
    # 4-d, broadcast along two axes, only one gradient asked for
    a4, b4, g4 = seeded((3, 1, 5, 7), 4, -1, 1), seeded((3, 6, 1, 7), 5, -1, 1), seeded((3, 6, 5, 7), 6, -1, 1)
    _, (da4_r,) = ref_exec(ref, cmd, None, 0, [g4, a4, b4], [np.zeros_like(a4)])
    st, (da4_g,) = gpu_exec(nnc, cmd, None, 0, [g4, a4, b4], [np.zeros_like(a4)])
    assert st == 0
    assert_close(da4_g, da4_r, 1e-5, "da 4-d")


@pytest.mark.parametrize("broadcast_w,with_bias", [(False, False), (True, False), (False, True), (True, True)])
def test_gemm_two_batch_axes(gpu, ref, broadcast_w, with_bias):
    """test/int/nnc/cublas.tests.c:1799-2228: a [2, 4, 10, 128] x w^T [2, 4, 64, 128] (or a shared [64, 128]) -> b [2, 4, 10, 64],
    forward and backward (shared dw / dbias accumulate over both batch axes)"""
    nnc = gpu
    a = seeded((2, 4, 10, 128), 1, -1, 1)
    w = seeded((64, 128) if broadcast_w else (2, 4, 64, 128), 2, -1, 1) / 11.0
    bias = seeded((64,), 3, -1, 1) if with_bias else None
    tb = (0, 1) if broadcast_w else (2, 3)
    fwd = nnc.CMD_GEMM_FORWARD((0, 0), tb)
    ins = [a, w] + ([bias] if with_bias else [])
    _, (b_r,) = ref_exec(ref, fwd, None, 0, ins, [np.zeros((2, 4, 10, 64), np.float32)])
    st, (b_g,) = gpu_exec(nnc, fwd, None, 0, ins, [np.zeros((2, 4, 10, 64), np.float32)])
    assert st == 0
    assert_close(b_g, b_r, 2e-5, "forward")
    g = seeded((2, 4, 10, 64), 4, -1, 1)
    bwd = nnc.CMD_GEMM_BACKWARD((0, 0), tb)
    outs = lambda: [np.zeros_like(a), np.zeros_like(w)] + ([np.zeros((64,), np.float32)] if with_bias else [])
    _, outs_r = ref_exec(ref, bwd, None, 0, [g, a, w], outs())
    st, outs_g = gpu_exec(nnc, bwd, None, 0, [g, a, w], outs())
    assert st == 0
    for name, x, y in zip(("h", "dw", "dbias"), outs_g, outs_r):
        assert_close(x, y, 5e-5, name)


def test_set_every_datatype(gpu):
    nnc = gpu
    for np_t, dt in ((np.float64, abi.CCV_64F), (np.float32, abi.CCV_32F), (np.int32, abi.CCV_32S)):
        t = nnc.gpu_tensor([11, 10, 9, 8], NHWC, dt)
        assert nnc.cmd_exec(nnc.CMD_SET_FORWARD(10), None, 0, [], [t], None) == 0
        out = t.download()
        t.free()
        assert out.dtype == np_t and np.array_equal(out, np.full((11, 10, 9, 8), 10, np_t))
    for kind in (abi.CCV_16BF, abi.CCV_16F):
        st, (out,) = gpu_exec16(nnc, nnc.CMD_SET_FORWARD(-1.5), None, 0, [], [np.zeros((7, 33), np.float32)], kind)
        assert st == 0 and np.array_equal(out, np.full((7, 33), -1.5, np.float32))


def test_ewsum_int32(gpu):
    nnc = gpu
    r = np.random.RandomState(1)
    xs = [r.randint(-1000, 1000, size=(17, 33)).astype(np.int32) for _ in range(3)]
    st, (out,) = gpu_exec(nnc, nnc.CMD_EWSUM_FORWARD(), None, 0, xs, [np.zeros((17, 33), np.int32)])
    assert st == 0 and np.array_equal(out, xs[0] + xs[1] + xs[2])


@pytest.mark.parametrize("kind", [abi.CCV_16F, abi.CCV_16BF])
def test_fp32_only_commands_on_16bit_tensors(gpu, ref, kind):
    """softmax / add / mul / scalar mul / softmax cross-entropy on half tensors (test/int/nnc/cudnn.tests.c:3504-3678, 4151-4323,
    4363-4735): functional form (widen, fp32 command, one rounding); oracle = CPU_REF on the rounded inputs, <= 1e-2"""
    nnc = gpu
    x, y = round16(seeded((10, 100), 1, -1, 1), kind), round16(seeded((10, 100), 2, -1, 1), kind)
    z = lambda: np.zeros((10, 100), np.float32)
    for name, cmd, ins in (("softmax", nnc.CMD_SOFTMAX_FORWARD(), [x]), ("add", nnc.CMD_ADD_FORWARD(0.5, 0.2), [x, y]), ("mul", nnc.CMD_MUL_FORWARD(0.7), [x, y]),
                           ("scalar mul", nnc.CMD_SCALAR_MUL_FORWARD(0.3), [x])):
        _, (o_r,) = ref_exec(ref, cmd, None, 0, ins, [z()])
        st, (o_g,) = gpu_exec16(nnc, cmd, None, 0, ins, [z()], kind)
        assert st == 0, name
        assert_close(o_g, o_r, 1e-2, name)
    g = round16(seeded((10, 100), 3, -1, 1), kind)
    _, (p_r,) = ref_exec(ref, nnc.CMD_SOFTMAX_FORWARD(), None, 0, [x], [z()], whole=True)  # the backward's operand is made from it
    p16 = round16(p_r, kind)
    _, (h_r,) = ref_exec(ref, nnc.CMD_SOFTMAX_BACKWARD(), None, 0, [g, None, p16], [z()])
    st, (h_g,) = gpu_exec16(nnc, nnc.CMD_SOFTMAX_BACKWARD(), None, 0, [g, None, p16], [z()], kind)
    assert st == 0
    assert_close(h_g, h_r, 1e-2, "softmax backward")
    # fused softmax + cross entropy with int32 labels: loss c [10, 1], probabilities d [10, 100]
    label = np.random.RandomState(7).randint(0, 100, size=(10,)).astype(np.int32)
    _, (c_r, d_r) = ref_exec(ref, nnc.CMD_SOFTMAX_CROSSENTROPY_FORWARD(), None, 0, [x, label], [np.zeros((10, 1), np.float32), z()])
    st, (c_g, d_g) = gpu_exec16(nnc, nnc.CMD_SOFTMAX_CROSSENTROPY_FORWARD(), None, 0, [x, label], [np.zeros((10, 1), np.float32), z()], kind)
    assert st == 0
    assert_close(c_g, c_r, 1e-2, "softmax cross-entropy loss"), assert_close(d_g, d_r, 1e-2, "softmax cross-entropy probabilities")


@pytest.mark.parametrize("which", ["max", "avg"])
def test_pooling_nchw(gpu, ref, which):
    """test/int/nnc/cudnn.tests.c:2772-2870: [C, H, W] = [10, 6, 6] NCHW, 2 x 2 stride 2; also 4-d with a border; backward"""
    nnc = gpu
    fwd = (nnc.CMD_MAX_POOL_FORWARD if which == "max" else nnc.CMD_AVERAGE_POOL_FORWARD)
    bwd = (nnc.CMD_MAX_POOL_BACKWARD if which == "max" else nnc.CMD_AVERAGE_POOL_BACKWARD)
    for shape_nhwc, k, stride, pad in (((6, 6, 10), 2, 2, 0), ((1, 9, 9, 16), 3, 2, 1)):  # one image: CPU_REF's pooling walks image 0 only
        x = seeded(shape_nhwc, 1, -1, 1)
        H = shape_nhwc[-3]
        P = (H + 2 * pad - k) // stride + 1
        out_nhwc = shape_nhwc[:-3] + (P, P, shape_nhwc[-1])
        hint = nnc.hint((stride, stride), (pad, pad))
        _, (y_r,) = ref_exec(ref, fwd(k, k), hint, 0, [x], [np.zeros(out_nhwc, np.float32)])
        perm = (2, 0, 1) if len(shape_nhwc) == 3 else (0, 3, 1, 2)
        back = (1, 2, 0) if len(shape_nhwc) == 3 else (0, 2, 3, 1)
        xc = np.ascontiguousarray(x.transpose(perm))
        st, (y_g,) = gpu_exec(nnc, fwd(k, k), hint, 0, [xc], [np.zeros(tuple(np.array(out_nhwc)[list(perm)]), np.float32)], fmt=NCHW)
        assert st == 0
        assert same(y_g.transpose(back), y_r) if which == "max" else max_abs_diff(y_g.transpose(back), y_r) <= 1e-6
        g = seeded(out_nhwc, 2, -1, 1)
        ins_r = [g, x, y_r] if which == "max" else [g]
        _, (h_r,) = ref_exec(ref, bwd(k, k), hint, 0, ins_r, [np.zeros(shape_nhwc, np.float32)])
        gc, yc = np.ascontiguousarray(g.transpose(perm)), y_g  # each side's backward reads its own forward output (compared above)
        ins_g = [gc, xc, yc] if which == "max" else [gc]
        st, (h_g,) = gpu_exec(nnc, bwd(k, k), hint, 0, ins_g, [np.zeros(xc.shape, np.float32)], fmt=NCHW)
        assert st == 0
        assert_close(h_g.transpose(back), h_r, 1e-6, which + " pool backward NCHW")


@pytest.mark.parametrize("nesterov", [0, 1])
def test_sgd_with_16bit_parameters(gpu, ref, nesterov):
    """test/int/nnc/sgd.tests.c:73-137, 250-314: g, a, m -> b, n all in half precision"""
    nnc = gpu
    kind = abi.CCV_16F
    g, a, m = round16(seeded((10, 100), 1, -1, 1), kind), round16(seeded((10, 100), 2, -1, 1), kind), round16(seeded((10, 100), 3, -1, 1), kind)
    cmd = nnc.CMD_SGD_FORWARD(nesterov, 0.002, 0.5, 0.9, 0.9, 0.0 if nesterov else 0.9)
    _, (b_r, n_r) = ref_exec(ref, cmd, None, 0, [g, a, m], [np.zeros_like(a), np.zeros_like(m)])
    st, (b_g, n_g) = gpu_exec16(nnc, cmd, None, 0, [g, a, m], [np.zeros_like(a), np.zeros_like(m)], kind)
    assert st == 0
    assert_close(b_g, b_r, 1e-3, "b"), assert_close(n_g, n_r, 1e-3, "n")


@pytest.mark.parametrize("half", [False, True])
def test_grouped_convolution_on_tensor_cores(gpu, ref, half):
    """groups = 2 with 32-wide groups: each group's channel slices are made dense and run on the tcgen05 kernels (forward, filter and
    data gradients); CPU_REF's grouped NHWC path is the oracle (convolution/ccv_nnc_conv_cpu_ref.c:47-65).  Half precision: oracle on
    the rounded inputs (there is no 16-bit FFMA fallback, so this also proves the tensor-core path took it)."""
    nnc = gpu
    N, H, C, K, R, groups = 2, 12, 64, 64, 3, 2
    x, w, bias = seeded((N, H, H, C), 1, -1, 1), seeded((K, R, R, C // groups), 2, -1, 1) / (R * R * C // groups) ** 0.5, seeded((K,), 3, -1, 1)
    g = seeded((N, H, H, K), 4, -1, 1)
    kind = abi.CCV_16F
    if half:
        x, w, bias, g = (round16(t, kind) for t in (x, w, bias, g))
    hint = nnc.hint((1, 1), (1, 1))
    fwd, bwd = nnc.CMD_CONVOLUTION_FORWARD(groups, K, R, R, C), nnc.CMD_CONVOLUTION_BACKWARD(groups, K, R, R, C)
    _, (y_r,) = ref_exec(ref, fwd, hint, 0, [x, w, bias], [np.zeros((N, H, H, K), np.float32)])
    _, (h_r, dw_r, db_r) = ref_exec(ref, bwd, hint, 0, [g, x, w], [np.zeros_like(x), np.zeros_like(w), np.zeros_like(bias)])
    if half:
        st, (y_g,) = gpu_exec16(nnc, fwd, hint, 0, [x, w, bias], [np.zeros((N, H, H, K), np.float32)], kind)
        outs = [np.zeros_like(x), np.zeros_like(w), np.zeros_like(bias)]
        st2, (h_g, dw_g, db_g) = gpu_exec16(nnc, bwd, hint, 0, [g, x, w], outs, kind)
    else:
        st, (y_g,) = gpu_exec(nnc, fwd, hint, 0, [x, w, bias], [np.zeros((N, H, H, K), np.float32)])
        st2, (h_g, dw_g, db_g) = gpu_exec(nnc, bwd, hint, 0, [g, x, w], [np.zeros_like(x), np.zeros_like(w), np.zeros_like(bias)])
    assert st == 0 and st2 == 0
    tol = 1e-2 if half else 1e-3
    for name, a, b in (("y", y_g, y_r), ("h", h_g, h_r), ("dw", dw_g, dw_r), ("dbias", db_g, db_r)):
        assert_close(a, b, tol, "grouped " + name)


def test_convolution_backward_half_three_channels(gpu, ref):
    """test/int/nnc/cudnn.tests.c:499-577: the 7 x 7 stride-2 stem in half precision, data gradient included (3-channel pixels:
    the tensor-core path cannot address them; functional form)"""
    nnc = gpu
    kind = abi.CCV_16F
    N, H, C, K, R = 2, 20, 3, 16, 7
    P = (H + 6 - R) // 2 + 1
    g, x, w = round16(seeded((N, P, P, K), 1, -1, 1), kind), round16(seeded((N, H, H, C), 2, -1, 1), kind), round16(seeded((K, R, R, C), 3, -1, 1) / 12.0, kind)
    cmd, hint = nnc.CMD_CONVOLUTION_BACKWARD(1, K, R, R, C), nnc.hint((2, 2), (3, 3))
    _, (h_r, dw_r, db_r) = ref_exec(ref, cmd, hint, 0, [g, x, w], [np.zeros_like(x), np.zeros_like(w), np.zeros((K,), np.float32)])
    st, (h_g, dw_g, db_g) = gpu_exec16(nnc, cmd, hint, 0, [g, x, w], [np.zeros_like(x), np.zeros_like(w), np.zeros((K,), np.float32)], kind)
    assert st == 0
    assert_close(h_g, h_r, 1e-2, "h"), assert_close(dw_g, dw_r, 1e-2, "dw"), assert_close(db_g, db_r, 1e-2, "dbias")


def test_gemm_with_a_matrix_as_third_operand(gpu):
    """test/int/nnc/cublas.tests.c:164-211: c = a b + d with d a full [4, 3] matrix (small integers: exact)"""
    nnc = gpu
    a = np.array([[1, 2], [3, 4], [5, 6], [7, 8]], np.float32)
    b = np.array([[7, 8, 9], [10, 11, 12]], np.float32)
    d = np.tile(np.array([1, -1, 1], np.float32), (4, 1))
    st, (c,) = gpu_exec(nnc, nnc.CMD_GEMM_FORWARD(), None, 0, [a, b, d], [np.zeros((4, 3), np.float32)])
    assert st == 0 and np.array_equal(c, a @ b + d)


@pytest.mark.parametrize("amsgrad", [0, 1])
def test_adam_forward(gpu, ref, amsgrad):
    """ADAM (L2 decay inside the gradient, adam/ccv_nnc_adam_cpu_ref.c:117-123) in fp32, and ADAMW with half-precision parameters and
    moments (test/int/nnc/adam.tests.c:300-360: <= 1e-3 against the fp32 CPU run on the rounded inputs)"""
    nnc = gpu
    shape = (10, 100)
    g, a, m, v, vm = seeded(shape, 1, -1, 1), seeded(shape, 2, -1, 1), seeded(shape, 3, -1, 1), seeded(shape, 4, 0, 1), seeded(shape, 5, 0, 1)
    cmd = nnc.CMD_ADAM_FORWARD(3, 0.002, 0.9, 0.98, 0.01, 1e-9, amsgrad)
    ins = [g, a, m, v] + ([vm] if amsgrad else [])
    outs = lambda: [np.zeros(shape, np.float32) for _ in range(4 if amsgrad else 3)]
    _, o_r = ref_exec(ref, cmd, None, 0, ins, outs())
    st, o_g = gpu_exec(nnc, cmd, None, 0, ins, outs())
    assert st == 0
    for x, y in zip(o_g, o_r):
        assert_close(x, y, 1e-5, "adam")
    kind = abi.CCV_16F
    ins16 = [round16(t, kind) for t in ins]
    cmdw = nnc.CMD_ADAMW_FORWARD(3, 0.002, 0.9, 0.98, 0.01, 1e-9, amsgrad)
    _, ow_r = ref_exec(ref, cmdw, None, 0, ins16, outs())
    st, ow_g = gpu_exec16(nnc, cmdw, None, 0, ins16, outs(), kind)
    assert st == 0
    for x, y in zip(ow_g, ow_r):
        assert_close(x, y, 2e-3, "adamw half")
