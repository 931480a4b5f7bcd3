"""SURVEY.md 8f-4: the commands a transformer block around SDPA needs -- GELU, SWISH, INDEX_SELECT, ADAMW -- on
CCV_NNC_BACKEND_GPU_SM100 against the reference's CPU_REF (gelu/ccv_nnc_gelu_cpu_ref.c, swish/..., index/ccv_nnc_index_select_cpu_ref.c,
adam/ccv_nnc_adamw_cpu_ref.c).  fp32 <= 1e-5 (same formulas, fp32 libm vs device intrinsics); bf16 through the rounded-input
protocol <= 1e-2; INDEX_SELECT is a copy: bit-exact, its backward adds rows in index order: bit-exact on integer-valued data."""
import numpy as np
import pytest

from ccv_b200 import abi
from tests.util import assert_close, gpu_exec, gpu_exec16, ref_exec, round16, same, seeded

pytestmark = [pytest.mark.gpu, pytest.mark.ref]


@pytest.mark.parametrize("name,tanh", [("gelu", 0), ("gelu", 1), ("swish", 0)])
def test_gelu_swish_forward_backward(gpu, ref, name, tanh):
    nnc = gpu
    shape = (6, 37, 129)  # odd sizes: vector body + scalar tail
    x, g = seeded(shape, 1, -4, 4), seeded(shape, 2, -1, 1)
    if name == "gelu":
        fwd, bwd = nnc.CMD_GELU_FORWARD(tanh), nnc.CMD_GELU_BACKWARD(tanh)
    else:
        fwd, bwd = nnc.CMD_SWISH_FORWARD(), nnc.CMD_SWISH_BACKWARD()
    _, (y_r,) = ref_exec(ref, fwd, None, 0, [x], [np.zeros(shape, np.float32)])
    st, (y_g,) = gpu_exec(nnc, fwd, None, 0, [x], [np.zeros(shape, np.float32)])
    assert st == 0
    assert_close(y_g, y_r, 1e-5, name + " forward")
    ins = [g, x, y_r]
    _, (h_r,) = ref_exec(ref, bwd, None, 0, ins, [np.zeros(shape, np.float32)])
    st, (h_g,) = gpu_exec(nnc, bwd, None, 0, ins, [np.zeros(shape, np.float32)])
    assert st == 0
    assert_close(h_g, h_r, 1e-5, name + " backward")
    # bf16 tensors: oracle on the rounded inputs
    xb, gb = round16(x, abi.CCV_16BF), round16(g, abi.CCV_16BF)
    _, (yb_r,) = ref_exec(ref, fwd, None, 0, [xb], [np.zeros(shape, np.float32)])
    st, (yb_g,) = gpu_exec16(nnc, fwd, None, 0, [xb], [np.zeros(shape, np.float32)], abi.CCV_16BF)
    assert st == 0
    assert_close(yb_g, yb_r, 1e-2, name + " forward bf16")
    _, (hb_r,) = ref_exec(ref, bwd, None, 0, [gb, xb, yb_r], [np.zeros(shape, np.float32)])
    st, (hb_g,) = gpu_exec16(nnc, bwd, None, 0, [gb, xb, yb_g], [np.zeros(shape, np.float32)], abi.CCV_16BF)
    assert st == 0
    assert_close(hb_g, hb_r, 1e-2, name + " backward bf16")


def test_index_select_forward_backward(gpu, ref):
    nnc = gpu
    rows, cols, n = 50, 96, 33
    a = seeded((rows, cols), 1, -1, 1)
    idx = np.random.RandomState(3).randint(0, rows, size=(n,)).astype(np.int32)
    idx[:4] = [7, 7, 0, rows - 1]  # repeated rows: the backward must accumulate them
    _, (b_r,) = ref_exec(ref, nnc.CMD_INDEX_SELECT_FORWARD(), None, 0, [a, idx], [np.zeros((n, cols), np.float32)])
    st, (b_g,) = gpu_exec(nnc, nnc.CMD_INDEX_SELECT_FORWARD(), None, 0, [a, idx], [np.zeros((n, cols), np.float32)])
    assert st == 0 and same(b_g, b_r) and np.array_equal(b_g, a[idx])
    g = np.round(seeded((n, cols), 2, -8, 8)).astype(np.float32)  # integer-valued: the sum is exact in any order
    _, (h_r,) = ref_exec(ref, nnc.CMD_INDEX_SELECT_BACKWARD(), None, 0, [g, None, idx], [np.zeros((rows, cols), np.float32)])
    st, (h_g,) = gpu_exec(nnc, nnc.CMD_INDEX_SELECT_BACKWARD(), None, 0, [g, None, idx], [np.full((rows, cols), 5.0, np.float32)])
    assert st == 0 and same(h_g, h_r)
    # fp32 indices interpolate between neighbouring rows (index_select_cpu_ref.c:47-63)
    fidx = np.array([0.0, 0.25, 10.5, rows - 1.0, rows - 1.5], np.float32)
    _, (c_r,) = ref_exec(ref, nnc.CMD_INDEX_SELECT_FORWARD(), None, 0, [a, fidx], [np.zeros((5, cols), np.float32)])
    st, (c_g,) = gpu_exec(nnc, nnc.CMD_INDEX_SELECT_FORWARD(), None, 0, [a, fidx], [np.zeros((5, cols), np.float32)])
    assert st == 0
    assert_close(c_g, c_r, 1e-6, "interpolating index select")
    # bf16 rows are copied bit for bit
    ab = round16(a, abi.CCV_16BF)
    st, (bb_g,) = gpu_exec16(nnc, nnc.CMD_INDEX_SELECT_FORWARD(), None, 0, [ab, idx], [np.zeros((n, cols), np.float32)], abi.CCV_16BF)
    assert st == 0 and np.array_equal(bb_g, ab[idx])


@pytest.mark.parametrize("amsgrad", [0, 1])
@pytest.mark.parametrize("g_kind", [abi.CCV_32F, abi.CCV_16BF])
def test_adamw(gpu, ref, amsgrad, g_kind):
    nnc = gpu
    n = 10007
    g = seeded((n,), 1, -1, 1)
    if g_kind != abi.CCV_32F:
        g = round16(g, g_kind)
    a, m, v, vm = seeded((n,), 2, -1, 1), seeded((n,), 3, -0.1, 0.1), seeded((n,), 4, 0, 0.01), seeded((n,), 5, 0, 0.02)
    cmd = nnc.CMD_ADAMW_FORWARD(3, 0.01, 0.9, 0.999, 0.05, 1e-8, amsgrad, scale=0.5)
    ins = [g, a, m, v] + ([vm] if amsgrad else [])
    mk = lambda: [np.zeros_like(a), np.zeros_like(m), np.zeros_like(v)] + ([np.zeros_like(vm)] if amsgrad else [])
    _, outs_r = ref_exec(ref, cmd, None, 0, ins, mk())
    outs0 = mk()
    if g_kind == abi.CCV_32F:
        st, outs_g = gpu_exec(nnc, cmd, None, 0, ins, outs0)
    else:
        keep = {id(t) for t in ins[1:] + outs0}
        st, outs_g = gpu_exec16(nnc, cmd, None, 0, ins, outs0, g_kind, keep32=keep)
    assert st == 0, nnc.lib().ccv_nnc_sm100_last_error()
    for got, want, name in zip(outs_g, outs_r, ("parameters", "first moment", "second moment", "max second moment")):
        assert_close(got, want, 1e-5, name)
