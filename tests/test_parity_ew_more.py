"""The remaining element-wise / reduction commands (SURVEY.md 2.3, VERDICT r01 "missing" 8) on CCV_NNC_BACKEND_GPU_SM100 against the
reference's CPU_REF: SIGMOID, TANH, LEAKY_RELU, EWEXP, EWLOG, EWSQRT, CLAMP, EWDIV (forward / backward, also without a gradient),
REDUCE_SUM / MEAN / MAX / MIN / NORM2 (forward / backward over one, two and all axes) and MASKED_FILL (int32 and fp32 masks,
broadcast).  fp32 <= 1e-5 of max|ref| (same formulas; libm vs device intrinsics), sums <= 1e-5 (fp32 partial sums in another order),
bf16 through the rounded-input protocol <= 1e-2; CLAMP, LEAKY_RELU, MAX / MIN and MASKED_FILL are selections: bit-exact."""
import numpy as np
import pytest

from ccv_b200 import abi
from tests.util import assert_close, gpu_exec, gpu_exec16, max_abs, max_abs_diff, ref_exec, round16, same, seeded

pytestmark = [pytest.mark.gpu, pytest.mark.ref]
NAN = float("nan")
SHAPE = (5, 33, 67)  # odd sizes: vector body + scalar tail


def _z(shape=SHAPE):
    return np.zeros(shape, np.float32)


NUMPY = {  # the forward in float64, for an operand both sides are given
    "SIGMOID": lambda x: 1 / (1 + np.exp(-x)), "TANH": np.tanh, "LEAKY_RELU": lambda x: np.where(x > 0, x, 0.2 * x), "EWEXP": np.exp,
    "EWLOG": np.log, "EWSQRT": np.sqrt, "CLAMP": lambda x: np.clip(x, -0.5, 0.75),
}
UNARY = {
    # name: (forward ctor args, input range, which operand the backward reads: 1 = a, 2 = b)
    "SIGMOID": ((), (-6, 6), 2), "TANH": ((), (-3, 3), 2), "LEAKY_RELU": ((0.2,), (-2, 2), 2), "EWEXP": ((), (-3, 3), 2),
    "EWLOG": ((), (0.1, 5), 1), "EWSQRT": ((), (0.1, 5), 2), "CLAMP": ((-0.5, 0.75), (-2, 2), 2),
}


@pytest.mark.parametrize("name", sorted(UNARY))
def test_unary_forward_backward(gpu, ref, name):
    nnc = gpu
    args, (lo, hi), which = UNARY[name]
    fwd, bwd = getattr(nnc, "CMD_%s_FORWARD" % name)(*args), getattr(nnc, "CMD_%s_BACKWARD" % name)(*args)
    x, g = seeded(SHAPE, 1, lo, hi), seeded(SHAPE, 2, -1, 1)
    _, (y_r,) = ref_exec(ref, fwd, None, 0, [x], [_z()])
    st, (y_g,) = gpu_exec(nnc, fwd, None, 0, [x], [_z()])
    assert st == 0
    exact = name in ("CLAMP", "LEAKY_RELU")
    if exact:
        assert same(y_g, y_r), name
    else:
        assert_close(y_g, y_r, 1e-5, name + " forward")
    # each side's backward reads its own forward output (compared above)
    _, (h_r,) = ref_exec(ref, bwd, None, 0, [g, x, y_r] if which == 2 else [g, x], [_z()])
    st, (h_g,) = gpu_exec(nnc, bwd, None, 0, [g, x, y_g] if which == 2 else [g, x], [_z()])
    assert st == 0
    assert_close(h_g, h_r, 1e-5, name + " backward")
    if name == "EWEXP":
        # no incoming gradient = all ones (ew_cpu_ref.c:1043-1044; CPU_REF's sigmoid / tanh backward dereference g before testing it,
        # sigmoid_cpu_ref.c:44, so that form has no oracle there)
        _, (h0_r,) = ref_exec(ref, bwd, None, 0, [None, x, y_r], [_z()])
        st, (h0_g,) = gpu_exec(nnc, bwd, None, 0, [None, x, y_g], [_z()])
        assert st == 0
        assert_close(h0_g, h0_r, 1e-5, name + " backward without g")
    # bf16: oracle on rounded inputs
    xb, gb = round16(x, abi.CCV_16BF), round16(g, abi.CCV_16BF)
    _, (yb_r,) = ref_exec(ref, fwd, None, 0, [xb], [_z()])
    st, (yb_g,) = gpu_exec16(nnc, fwd, None, 0, [xb], [_z()], abi.CCV_16BF)
    assert st == 0
    assert_close(yb_g, yb_r, 1e-2, name + " forward bf16")
    yb = round16(NUMPY[name](xb.astype(np.float64)).astype(np.float32), abi.CCV_16BF)  # the bf16 forward output, as an operand
    insb = [gb, xb, yb] if which == 2 else [gb, xb]
    _, (hb_r,) = ref_exec(ref, bwd, None, 0, insb, [_z()])
    st, (hb_g,) = gpu_exec16(nnc, bwd, None, 0, insb, [_z()], abi.CCV_16BF)
    assert st == 0
    assert_close(hb_g, hb_r, 1e-2, name + " backward bf16")


def test_clamp_open_sides(gpu, ref):
    nnc = gpu
    x = seeded(SHAPE, 3, -2, 2)
    for lo, hi in ((NAN, 0.5), (-0.25, NAN)):
        _, (y_r,) = ref_exec(ref, nnc.CMD_CLAMP_FORWARD(lo, hi), None, 0, [x], [_z()])
        st, (y_g,) = gpu_exec(nnc, nnc.CMD_CLAMP_FORWARD(lo, hi), None, 0, [x], [_z()])
        assert st == 0 and same(y_g, y_r)
        g = seeded(SHAPE, 4, -1, 1)
        _, (h_r,) = ref_exec(ref, nnc.CMD_CLAMP_BACKWARD(lo, hi), None, 0, [g, x, y_r], [_z()])
        st, (h_g,) = gpu_exec(nnc, nnc.CMD_CLAMP_BACKWARD(lo, hi), None, 0, [g, x, y_r], [_z()])
        assert st == 0 and same(h_g, h_r)


def test_ewdiv_forward_backward(gpu, ref):
    nnc = gpu
    a, b, g = seeded(SHAPE, 1, -2, 2), seeded(SHAPE, 2, 0.5, 3), seeded(SHAPE, 3, -1, 1)
    _, (c_r,) = ref_exec(ref, nnc.CMD_EWDIV_FORWARD(), None, 0, [a, b], [_z()])
    st, (c_g,) = gpu_exec(nnc, nnc.CMD_EWDIV_FORWARD(), None, 0, [a, b], [_z()])
    assert st == 0
    assert_close(c_g, c_r, 1e-6, "a / b")
    _, (r_r,) = ref_exec(ref, nnc.CMD_EWDIV_FORWARD(), None, 0, [None, b], [_z()])
    st, (r_g,) = gpu_exec(nnc, nnc.CMD_EWDIV_FORWARD(), None, 0, [None, b], [_z()])
    assert st == 0
    assert_close(r_g, r_r, 1e-6, "1 / b")
    _, (ha_r, hb_r) = ref_exec(ref, nnc.CMD_EWDIV_BACKWARD(), None, 0, [g, a, b, c_r], [_z(), _z()])
    st, (ha_g, hb_g) = gpu_exec(nnc, nnc.CMD_EWDIV_BACKWARD(), None, 0, [g, a, b, c_g], [_z(), _z()])  # each side's own quotient
    assert st == 0
    assert_close(ha_g, ha_r, 1e-5, "d(a / b) / da")
    assert_close(hb_g, hb_r, 1e-5, "d(a / b) / db")
    _, (ha1_r,) = ref_exec(ref, nnc.CMD_EWDIV_BACKWARD(), None, 0, [g, a, b, c_r], [_z()])
    st, (ha1_g,) = gpu_exec(nnc, nnc.CMD_EWDIV_BACKWARD(), None, 0, [g, a, b, c_r], [_z()])
    assert st == 0
    assert_close(ha1_g, ha1_r, 1e-5, "only d / da")


REDUCE_CASES = [((4, 6, 10, 33), (1,)), ((4, 6, 10, 33), (3,)), ((4, 6, 10, 33), (0, 2)), ((3, 700), (1,)), ((2, 3, 5000), (0, 1, 2)), ((17, 9, 4), (0,))]


@pytest.mark.parametrize("mode", ["SUM", "MEAN", "MAX", "MIN", "NORM2"])
@pytest.mark.parametrize("shape,axes", REDUCE_CASES)
def test_reduce_forward_backward(gpu, ref, mode, shape, axes):
    nnc = gpu
    fwd, bwd = getattr(nnc, "CMD_REDUCE_%s_FORWARD" % mode)(*axes), getattr(nnc, "CMD_REDUCE_%s_BACKWARD" % mode)(*axes)
    out_shape = tuple(1 if i in axes else d for i, d in enumerate(shape))
    x, g = seeded(shape, 1, -1, 1), seeded(out_shape, 2, -1, 1)
    _, (y_r,) = ref_exec(ref, fwd, None, 0, [x], [_z(out_shape)])
    st, (y_g,) = gpu_exec(nnc, fwd, None, 0, [x], [_z(out_shape)])
    assert st == 0
    if mode in ("MAX", "MIN"):
        assert same(y_g, y_r), mode
    else:
        # the bound is relative to the magnitude of what is summed, not of a sum that may cancel
        err = max_abs_diff(y_g, y_r) / max(np.abs(x).sum(axis=axes).max() * (1.0 / np.prod([shape[a] for a in axes]) if mode == "MEAN" else 1.0), 1e-30)
        assert err <= 1e-5 if mode != "NORM2" else max_abs_diff(y_g, y_r) <= 1e-5 * max_abs(y_r), (mode, err)
    _, (h_r,) = ref_exec(ref, bwd, None, 0, [g, x, y_r], [_z(shape)])
    st, (h_g,) = gpu_exec(nnc, bwd, None, 0, [g, x, y_g], [_z(shape)])  # each side's own forward output (compared above)
    assert st == 0
    assert_close(h_g, h_r, 1e-6, "reduce %s backward" % mode)
    if mode in ("SUM", "MEAN"):
        _, (h0_r,) = ref_exec(ref, bwd, None, 0, [None, x, y_r], [_z(shape)])
        st, (h0_g,) = gpu_exec(nnc, bwd, None, 0, [None, x, y_r], [_z(shape)])
        assert st == 0
        assert_close(h0_g, h0_r, 1e-6, "reduce %s backward without g" % mode)


def test_reduce_bf16(gpu, ref):
    nnc = gpu
    shape, axes, out_shape = (8, 40, 96), (1,), (8, 1, 96)
    x = round16(seeded(shape, 1, -1, 1), abi.CCV_16BF)
    for mode in ("SUM", "MEAN", "MAX", "NORM2"):
        fwd = getattr(nnc, "CMD_REDUCE_%s_FORWARD" % mode)(*axes)
        _, (y_r,) = ref_exec(ref, fwd, None, 0, [x], [_z(out_shape)])
        st, (y_g,) = gpu_exec16(nnc, fwd, None, 0, [x], [_z(out_shape)], abi.CCV_16BF)
        assert st == 0
        assert_close(y_g, y_r, 1e-2, "reduce %s bf16" % mode)


@pytest.mark.parametrize("mask_dtype", [np.int32, np.float32])
def test_masked_fill(gpu, ref, mask_dtype):
    nnc = gpu
    shape, mshape = (3, 5, 7, 19), (1, 5, 1, 19)  # the mask broadcasts over two axes
    a, g = seeded(shape, 1, -1, 1), seeded(shape, 2, -1, 1)
    mask = (np.random.RandomState(5).randint(0, 3, size=mshape)).astype(mask_dtype)
    fwd, bwd = nnc.CMD_MASKED_FILL_FORWARD(2, -1e9), nnc.CMD_MASKED_FILL_BACKWARD(2, -1e9)
    _, (c_r,) = ref_exec(ref, fwd, None, 0, [a, mask], [_z(shape)])
    st, (c_g,) = gpu_exec(nnc, fwd, None, 0, [a, mask], [_z(shape)])
    assert st == 0 and same(c_g, c_r)
    assert (c_g == -1e9).sum() == (np.broadcast_to(mask, shape) == 2).sum()
    _, (h_r,) = ref_exec(ref, bwd, None, 0, [g, None, mask], [_z(shape)])
    st, (h_g,) = gpu_exec(nnc, bwd, None, 0, [g, None, mask], [_z(shape)])
    assert st == 0 and same(h_g, h_r)


@pytest.mark.parametrize("n", [100003, 4096])
def test_random_uniform_and_normal(gpu, n):
    """RANDOM_UNIFORM / RANDOM_NORMAL (rand/gpu/ccv_nnc_rand_uniform_gpu_ref.cu:33-66): the contract is the distribution and a fresh seed
    per call from the stream context's generator (the protocol of test/int/nnc/random.tests.c: moments of a large sample)."""
    nnc = gpu
    st, (u1,) = gpu_exec(nnc, nnc.CMD_RANDOM_UNIFORM_FORWARD(-2.0, 3.0), None, 0, [], [np.zeros((n,), np.float32)])
    st2, (u2,) = gpu_exec(nnc, nnc.CMD_RANDOM_UNIFORM_FORWARD(-2.0, 3.0), None, 0, [], [np.zeros((n,), np.float32)])
    assert st == 0 and st2 == 0
    assert u1.min() >= -2.0 and u1.max() <= 3.0 and not np.array_equal(u1, u2)
    tol = 6.0 / np.sqrt(n)
    assert abs(u1.mean() - 0.5) <= 5 * tol / np.sqrt(12) * 1.0 + 1e-3 and abs(u1.std() - 5 / np.sqrt(12)) <= 0.05
    assert len(np.unique(u1)) > 0.95 * n
    st, (g1,) = gpu_exec(nnc, nnc.CMD_RANDOM_NORMAL_FORWARD(2.0, 1.0), None, 0, [], [np.zeros((n,), np.float32)])
    assert st == 0 and np.isfinite(g1).all()
    assert abs(g1.mean() - 1.0) <= 2 * tol + 1e-3 and abs(g1.std() - 2.0) <= 0.1
    # bf16 tensors
    st, (ub,) = gpu_exec16(nnc, nnc.CMD_RANDOM_UNIFORM_FORWARD(0.0, 1.0), None, 0, [], [np.zeros((n,), np.float32)], abi.CCV_16BF)
    assert st == 0 and ub.min() >= 0.0 and ub.max() <= 1.0 and abs(ub.mean() - 0.5) <= 0.02


@pytest.mark.xfail(strict=False, reason="DROPOUT was added after the builder's GPU budget was spent: first hardware run is the driver's")
@pytest.mark.parametrize("entirety", [0, 1])
def test_dropout_forward_backward(gpu, entirety):
    """DROPOUT (dropout/ccv_nnc_dropout_cpu_ref.c:16-215): b = mask ? 0 : a / (1 - p) with a byte mask in the reserved second output
    (dropout/ccv_nnc_dropout.c:21-44), backward h = mask ? 0 : g / (1 - p) with the same mask.  The random stream is this backend's
    (Philox keyed by the stream context's seed), so what is checked is what the reference's own tests check: the drop rate and the
    consistency of output, mask and gradient (test/int/nnc/cudnn.tests.c:3389-3464)."""
    nnc = gpu
    n, p = 20 * 50 * 100, 0.2
    a, g = seeded((20, 50, 100), 1, 0.5, 1.5), seeded((20, 50, 100), 2, 0.5, 1.5)
    mask_shape = (32, ((20 + 127) // 128) * 50 * 100) if not entirety else (1,)   # the reference's tensor_auto: 128-byte lines
    st, (b, mask) = gpu_exec(nnc, nnc.CMD_DROPOUT_FORWARD(p, entirety), None, 0, [a], [np.zeros_like(a), np.zeros(mask_shape, np.float32)])
    assert st == 0
    if entirety:
        dropped = bool(mask.view(np.int32)[0])
        assert np.array_equal(b, np.zeros_like(a)) if dropped else np.allclose(b, a / (1 - p), rtol=1e-6)
        m = np.full(a.shape, dropped)
    else:
        m = mask.view(np.uint8).reshape(-1)[:n].reshape(a.shape).astype(bool)
        assert abs(m.mean() - p) < 0.01
        assert np.array_equal(b == 0, m) and np.allclose(b[~m], (a / (1 - p))[~m], rtol=1e-6)
    st, (h,) = gpu_exec(nnc, nnc.CMD_DROPOUT_BACKWARD(p, entirety), None, 0, [g, None, None, None, mask], [np.zeros_like(g)])
    assert st == 0
    assert np.array_equal(h == 0, m) and np.allclose(h[~m], (g / (1 - p))[~m], rtol=1e-6)
