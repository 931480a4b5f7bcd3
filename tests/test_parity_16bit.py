"""The 16-bit (bf16 / fp16) datapath -- BASELINE.json configs[3], the dtype bin/nnc/imagenet.c:344 trains in -- against the
reference's CCV_NNC_BACKEND_CPU_REF.  CPU_REF has no 16-bit kernels for these commands (SURVEY.md 8c: "unpinned"), so the
protocol is the one the north star states: the oracle runs in fp32 on the inputs ROUNDED to the 16-bit type (what the GPU
tensors actually hold), the GPU result (fp32 accumulation, one rounding on the way out) is widened back and held to <= 1e-2
of max|ref|.  bf16 has 8 mantissa bits: one output rounding is already 2^-9 = 2e-3 relative."""
import numpy as np
import pytest

from ccv_b200 import abi
from tests.util import assert_close, gpu_exec16, ref_exec, round16, same, seeded

pytestmark = [pytest.mark.gpu, pytest.mark.ref]
KINDS = [abi.CCV_16BF, abi.CCV_16F]
TOL = 1e-2


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("M,N,K,ta,tb,with_bias", [(128, 128, 64, 0, 0, 0), (256, 192, 160, 0, 1, 1), (200, 136, 104, 1, 0, 1), (96, 72, 48, 1, 1, 0), (64, 1000, 2048, 0, 1, 1), (8, 64, 128, 0, 1, 0),
                                                      (4, 10, 2048, 0, 1, 1), (33, 17, 21, 0, 1, 1)])  # strides TMA cannot take: widened, multiplied in fp32, narrowed
def test_gemm_16bit_forward_backward(gpu, ref, kind, M, N, K, ta, tb, with_bias):
    nnc = gpu
    a = round16(seeded((K, M) if ta else (M, K), 11, -1, 1), kind)
    w = round16(seeded((N, K) if tb else (K, N), 12, -1, 1), kind)
    bias = round16(seeded((N,), 13), kind) if with_bias else None
    cmd = lambda c: c((0, 1) if ta else (0, 0), (0, 1) if tb else (0, 0))
    ins = [a, w] + ([bias] if with_bias else [])
    _, (b_ref,) = ref_exec(ref, cmd(nnc.CMD_GEMM_FORWARD), None, 0, ins, [np.zeros((M, N), np.float32)])
    st, (b_gpu,) = gpu_exec16(nnc, cmd(nnc.CMD_GEMM_FORWARD), None, 0, ins, [np.zeros((M, N), np.float32)], kind)
    assert st == 0, nnc.lib().ccv_nnc_sm100_last_error()
    assert_close(b_gpu, b_ref, TOL, "forward")
    g = round16(seeded((M, N), 14, -1, 1), kind)
    outs = lambda: [np.zeros_like(a), np.zeros_like(w), np.zeros((N,), np.float32)]
    _, (h_r, dw_r, db_r) = ref_exec(ref, cmd(nnc.CMD_GEMM_BACKWARD), None, 0, [g, a, w], outs())
    st, (h_g, dw_g, db_g) = gpu_exec16(nnc, cmd(nnc.CMD_GEMM_BACKWARD), None, 0, [g, a, w], outs(), kind)
    assert st == 0, nnc.lib().ccv_nnc_sm100_last_error()
    assert_close(h_g, h_r, TOL, "h"), assert_close(dw_g, dw_r, TOL, "dw"), assert_close(db_g, db_r, TOL, "dbias")


CONVS = [
    # (N, H, W, C, K, R, stride, pad, bias)
    (2, 12, 12, 64, 64, 3, 1, 1, 1), (2, 13, 9, 64, 128, 3, 2, 1, 1), (3, 14, 14, 64, 256, 1, 1, 0, 1), (2, 14, 14, 128, 64, 1, 2, 0, 0),
    (2, 16, 16, 32, 32, 3, 1, 1, 1),   # the stem's 32-channel layers: half of each 128-byte operand span is padding
    (2, 16, 16, 32, 64, 3, 1, 1, 0),
    (2, 16, 16, 3, 32, 3, 2, 1, 0),    # 3-channel stem: explicit im2col + GEMM
    (1, 20, 20, 16, 24, 7, 2, 3, 1), (4, 7, 7, 512, 2048, 1, 1, 0, 0), (4, 7, 7, 2048, 512, 1, 1, 0, 1),
]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N,H,W,C,K,R,st,pad,with_bias", CONVS)
def test_convolution_16bit_forward_backward(gpu, ref, kind, N, H, W, C, K, R, st, pad, with_bias):
    nnc = gpu
    P, Q = (H + 2 * pad - R) // st + 1, (W + 2 * pad - R) // st + 1
    a = round16(seeded((N, H, W, C), 21, -1, 1), kind)
    w = round16(seeded((K, R, R, C), 22, -1, 1) / (C * R * R) ** 0.5, kind)
    bias = round16(np.arange(K, dtype=np.float32) / K, kind) if with_bias else None
    hint = nnc.hint((st, st), (pad, pad))
    ins = [a, w] + ([bias] if with_bias else [])
    fwd, bwd = nnc.CMD_CONVOLUTION_FORWARD(1, K, R, R, C), nnc.CMD_CONVOLUTION_BACKWARD(1, K, R, R, C)
    _, (b_r,) = ref_exec(ref, fwd, hint, 0, ins, [np.zeros((N, P, Q, K), np.float32)])
    stt, (b_g,) = gpu_exec16(nnc, fwd, hint, 0, ins, [np.zeros((N, P, Q, K), np.float32)], kind)
    assert stt == 0, nnc.lib().ccv_nnc_sm100_last_error()
    assert_close(b_g, b_r, TOL, "forward")
    g = round16(seeded((N, P, Q, K), 23, -1, 1), kind)
    need_dx = C % 8 == 0
    outs = lambda: [np.zeros_like(a) if need_dx else None, np.zeros_like(w), np.zeros((K,), np.float32)]
    _, (h_r, dw_r, db_r) = ref_exec(ref, bwd, hint, 0, [g, a, w], [np.zeros_like(a), np.zeros_like(w), np.zeros((K,), np.float32)])
    stt, (h_g, dw_g, db_g) = gpu_exec16(nnc, bwd, hint, 0, [g, a, w], outs(), kind)
    assert stt == 0, nnc.lib().ccv_nnc_sm100_last_error()
    if need_dx:
        assert_close(h_g, h_r, TOL, "dgrad")
    assert_close(dw_g, dw_r, TOL, "wgrad"), assert_close(db_g, db_r, TOL, "dbias")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", [(8, 14, 14, 64), (4, 7, 7, 2048), (16, 28, 28, 32)])
def test_batch_norm_16bit(gpu, ref, kind, shape):
    """x / y / g / dx 16-bit; scale, bias, running and saved statistics, dscale, dbias fp32 (ccv_cnnp_model_addons.c:954-956)."""
    nnc = gpu
    C = shape[-1]
    x = round16(seeded(shape, 1, -2, 3), kind)
    scale, bias = seeded((1, 1, 1, C), 2, 0.5, 1.5), seeded((1, 1, 1, C), 3, -1, 1)
    mean_r, var_r = np.zeros((1, 1, 1, C), np.float32), np.ones((1, 1, 1, C), np.float32)
    mean_g, var_g = mean_r.copy(), var_r.copy()
    y_r, sm_r, sis_r = np.zeros(shape, np.float32), np.zeros((1, 1, 1, C), np.float32), np.zeros((1, 1, 1, C), np.float32)
    bn = nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9)
    assert ref_exec(ref, bn, None, 0, [x, scale, bias, mean_r, var_r], [y_r, mean_r, var_r, sm_r, sis_r])[0] == 0
    y0, sm0, sis0 = np.zeros(shape, np.float32), np.zeros((1, 1, 1, C), np.float32), np.zeros((1, 1, 1, C), np.float32)
    keep = {id(v) for v in (scale, bias, mean_g, var_g, sm0, sis0)}
    st, (y_g, mean_o, var_o, sm_g, sis_g) = gpu_exec16(nnc, bn, None, 0, [x, scale, bias, mean_g, var_g], [y0, mean_g, var_g, sm0, sis0], kind, keep32=keep)
    assert st == 0, nnc.lib().ccv_nnc_sm100_last_error()
    assert_close(y_g, y_r, TOL, "y"), assert_close(sm_g, sm_r, 1e-4, "saved mean"), assert_close(sis_g, sis_r, 1e-3, "saved inv_std")
    assert_close(mean_o, mean_r, 1e-4, "running mean"), assert_close(var_o, var_r, 1e-3, "running var")
    g = round16(seeded(shape, 5, -1, 1), kind)
    bwd = nnc.CMD_BATCH_NORM_BACKWARD(1e-4, 0, 0.9)
    ins = [g] + [None] * 4 + [x, scale] + [None] * 6 + [sm_r, sis_r]
    dx_r, ds_r, db_r = np.zeros(shape, np.float32), np.zeros((1, 1, 1, C), np.float32), np.zeros((1, 1, 1, C), np.float32)
    assert ref_exec(ref, bwd, None, 0, ins, [dx_r, ds_r, db_r])[0] == 0
    dx0, ds0, db0 = np.zeros(shape, np.float32), np.zeros((1, 1, 1, C), np.float32), np.zeros((1, 1, 1, C), np.float32)
    ins_g = [g] + [None] * 4 + [x, scale] + [None] * 6 + [sm_g, sis_g]  # each side's own saved statistics (compared above)
    keep = {id(v) for v in (scale, sm_g, sis_g, ds0, db0)}
    st, (dx_g, ds_g, db_g) = gpu_exec16(nnc, bwd, None, 0, ins_g, [dx0, ds0, db0], kind, keep32=keep)
    assert st == 0, nnc.lib().ccv_nnc_sm100_last_error()
    assert_close(dx_g, dx_r, TOL, "dx"), assert_close(ds_g, ds_r, 1e-3, "dscale"), assert_close(db_g, db_r, 1e-3, "dbias")


@pytest.mark.parametrize("kind", KINDS)
def test_relu_ewsum_pools_16bit(gpu, ref, kind):
    nnc = gpu
    shape = (4, 15, 15, 32)
    a, b = round16(seeded(shape, 1, -1, 1), kind), round16(seeded(shape, 2, -1, 1), kind)
    _, (r_r,) = ref_exec(ref, nnc.CMD_RELU_FORWARD(), None, 0, [a], [np.zeros(shape, np.float32)])
    st, (r_g,) = gpu_exec16(nnc, nnc.CMD_RELU_FORWARD(), None, 0, [a], [np.zeros(shape, np.float32)], kind)
    assert st == 0 and same(r_g, r_r)  # exact: max(x, 0) of representable values
    _, (h_r,) = ref_exec(ref, nnc.CMD_RELU_BACKWARD(), None, 0, [b, None, r_r], [np.zeros(shape, np.float32)])
    st, (h_g,) = gpu_exec16(nnc, nnc.CMD_RELU_BACKWARD(), None, 0, [b, None, r_g], [np.zeros(shape, np.float32)], kind)  # r_g equals r_r (checked above)
    assert st == 0 and same(h_g, h_r)
    _, (s_r,) = ref_exec(ref, nnc.CMD_EWSUM_FORWARD(), None, 0, [a, b, r_r], [np.zeros(shape, np.float32)])
    st, (s_g,) = gpu_exec16(nnc, nnc.CMD_EWSUM_FORWARD(), None, 0, [a, b, r_g], [np.zeros(shape, np.float32)], kind)
    assert st == 0
    assert_close(s_g, s_r, TOL, "ewsum")
    for name, fwd, bwd, k, stv, pad in (("max", nnc.CMD_MAX_POOL_FORWARD, nnc.CMD_MAX_POOL_BACKWARD, 3, 2, 1), ("avg", nnc.CMD_AVERAGE_POOL_FORWARD, nnc.CMD_AVERAGE_POOL_BACKWARD, 2, 2, 0)):
        P = (shape[1] + 2 * pad - k) // stv + 1
        hint = nnc.hint((stv, stv), (pad, pad))
        # CPU_REF pooling walks one image per call (SURVEY.md 0.6); each image is compared on its own (normalised per image: no
        # looser than over the batch)
        y_r = [np.zeros((P, P, shape[3]), np.float32) for _ in range(shape[0])]
        for n in range(shape[0]):
            ref_exec(ref, fwd(k, k), hint, 0, [a[n]], [y_r[n]])
        st, (y_g,) = gpu_exec16(nnc, fwd(k, k), hint, 0, [a], [np.zeros((shape[0], P, P, shape[3]), np.float32)], kind)
        assert st == 0, name
        for n in range(shape[0]):
            assert_close(y_g[n], y_r[n], TOL, name + " pool forward")
        gy = round16(seeded(y_g.shape, 7, -1, 1), kind)
        # the backward reads each side's own forward output (compared above); a max of 16-bit values is itself a 16-bit value
        dx_r = [np.zeros(shape[1:], np.float32) for _ in range(shape[0])]
        for n in range(shape[0]):
            ref_exec(ref, bwd(k, k), hint, 0, [gy[n], a[n], y_r[n]], [dx_r[n]])
        st, (dx_g,) = gpu_exec16(nnc, bwd(k, k), hint, 0, [gy, a, y_g], [np.zeros(shape, np.float32)], kind)
        assert st == 0, name
        for n in range(shape[0]):
            assert_close(dx_g[n], dx_r[n], TOL, name + " pool backward")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("nesterov", [0, 1])
def test_sgd_mixed_precision(gpu, ref, kind, nesterov):
    """gradient 16-bit, parameters and momenta fp32 (the mixed form of sgd/gpu/ccv_nnc_sgd_gpu_ref.cu:71-74)."""
    nnc = gpu
    n = 10000
    g, a, m = round16(seeded((n,), 1, -1, 1), kind), seeded((n,), 2, -1, 1), seeded((n,), 3, -0.1, 0.1)
    cmd = nnc.CMD_SGD_FORWARD(nesterov, 0.1, 0.5, 1e-3, 0.9, 0.0 if nesterov else 0.1)
    _, (b_r, n_r) = ref_exec(ref, cmd, None, 0, [g, a, m], [np.zeros_like(a), np.zeros_like(m)])
    b0, n0 = np.zeros_like(a), np.zeros_like(m)
    st, (b_g, n_g) = gpu_exec16(nnc, cmd, None, 0, [g, a, m], [b0, n0], kind, keep32={id(a), id(m), id(b0), id(n0)})
    assert st == 0, nnc.lib().ccv_nnc_sm100_last_error()
    assert_close(b_g, b_r, 1e-6, "parameters"), assert_close(n_g, n_r, 1e-6, "momentum")
