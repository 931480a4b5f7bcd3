"""Parity of layer norm, group norm, rms norm and upsample (the ops that feed attention blocks / resampling) vs CPU_REF."""
import numpy as np
import pytest

from ccv_b200 import abi, nnc as _nnc
from tests.util import NCHW, NHWC, assert_close, gpu_exec, ref_exec, seeded

pytestmark = [pytest.mark.gpu, pytest.mark.ref]


def _lnorm(cmd_id, eps, affine, axes):
    c = _nnc._simple(cmd_id)
    for i, a in enumerate(axes):
        c.info.lnorm.axis[i] = a
    c.info.lnorm.count, c.info.lnorm.epsilon, c.info.lnorm.elementwise_affine = len(axes), eps, affine
    return c


def _rms(cmd_id, eps, axes):
    c = _nnc._simple(cmd_id)
    for i, a in enumerate(axes):
        c.info.rmsnorm.axis[i] = a
    c.info.rmsnorm.count, c.info.rmsnorm.epsilon = len(axes), eps
    return c


@pytest.mark.parametrize("shape,axes", [((6, 10, 64), (2,)), ((4, 3, 5, 40), (1, 2, 3)), ((32, 1000), (1,))])
def test_layer_norm_forward_backward(gpu, ref, shape, axes):
    """protocol of test/int/nnc/cudnn.tests.c layer norm cases: statistics over the trailing axes, affine scale/bias."""
    nnc = gpu
    x = seeded(shape, 1, -1, 1)
    rshape = tuple(1 if i in axes else d for i, d in enumerate(shape))
    pshape = tuple(d if i in axes else 1 for i, d in enumerate(shape))
    scale, bias = seeded(pshape, 2), seeded(pshape, 3)
    fwd = _lnorm(abi.CCV_NNC_LAYER_NORM_FORWARD, 1e-5, 1, axes)
    mk = lambda: [np.zeros(shape, np.float32), np.zeros(rshape, np.float32), np.zeros(rshape, np.float32)]
    st_r, (y_r, m_r, s_r) = ref_exec(ref, fwd, None, 0, [x, scale, bias], mk())
    st_g, (y_g, m_g, s_g) = gpu_exec(nnc, fwd, None, 0, [x, scale, bias], mk())
    assert st_r == 0 and st_g == 0
    assert_close(y_g, y_r, 1e-4, "y"), assert_close(m_g, m_r, 1e-5, "mean"), assert_close(s_g, s_r, 1e-4, "inv_std")
    g = seeded(shape, 4, -1, 1)
    bwd = _lnorm(abi.CCV_NNC_LAYER_NORM_BACKWARD, 1e-5, 1, axes)
    ins = [g, None, None, x, scale, None, None, m_r, s_r]
    mk = lambda: [np.zeros(shape, np.float32), np.zeros(pshape, np.float32), np.zeros(pshape, np.float32)]
    st_r, (h_r, ds_r, db_r) = ref_exec(ref, bwd, None, 0, ins, mk())
    st_g, (h_g, ds_g, db_g) = gpu_exec(nnc, bwd, None, 0, ins, mk())
    assert st_r == 0 and st_g == 0
    assert_close(h_g, h_r, 1e-3, "dx"), assert_close(ds_g, ds_r, 1e-3, "dscale"), assert_close(db_g, db_r, 1e-3, "dbias")


def _gnorm(cmd_id, group_axis, groups, eps, affine, reduce_axes):
    c = _nnc._simple(cmd_id)
    c.info.gnorm.group_axis, c.info.gnorm.groups, c.info.gnorm.epsilon, c.info.gnorm.elementwise_affine = group_axis, groups, eps, affine
    for i, a in enumerate(reduce_axes):
        c.info.gnorm.reduce_axis[i] = a
    c.info.gnorm.reduce_count = len(reduce_axes)
    return c


@pytest.mark.parametrize("shape,group_axis,groups,reduce_axes,affine", [
    ((2, 16, 6, 5), 1, 4, (2, 3), 1),      # NCHW, test/unit/nnc/group.norm.tests.c: groups over channels, reduce over H, W
    ((2, 6, 5, 16), 3, 4, (1, 2), 1),      # NHWC
    ((3, 32, 7, 7), 1, 8, (2, 3), 0),      # no affine
    ((4, 24, 10), 1, 3, (2,), 1),          # 3-d
    ((2, 16, 2, 10), 1, 4, (), 1),         # test/int/nnc/cudnn.tests.c:1491-1560: statistics over the 4 channels of a group only (small variances: the epsilon word matters)
])
def test_group_norm_forward_backward(gpu, ref, shape, group_axis, groups, reduce_axes, affine):
    """norm/ccv_nnc_group_norm_cpu_ref.c: statistics per (sample, group); per-channel scale / bias.  CPU_REF (and the
    reference's GPU implementation) read the epsilon through the lnorm arm of the parameter union (:46), i.e. the integer
    reduce_count reinterpreted as a float (a denormal ~ 0) instead of gnorm.epsilon; the backend reads the same word."""
    nnc = gpu
    x = seeded(shape, 1, -1, 1)
    rshape = tuple(groups if i == group_axis else (1 if i in reduce_axes else d) for i, d in enumerate(shape))
    pshape = tuple(d if i == group_axis else 1 for i, d in enumerate(shape))
    if not reduce_axes:
        pshape = (1,) + tuple(shape[1:])  # the reference's own test shape: scale / bias per element of a sample
    scale, bias = seeded(pshape, 2), seeded(pshape, 3)
    fwd = _gnorm(abi.CCV_NNC_GROUP_NORM_FORWARD, group_axis, groups, 1e-5, affine, reduce_axes)
    mk = lambda: [np.zeros(shape, np.float32), np.zeros(rshape, np.float32), np.zeros(rshape, np.float32)]
    fin = [x, scale, bias] if affine else [x]
    st_r, (y_r, m_r, s_r) = ref_exec(ref, fwd, None, 0, fin, mk())
    st_g, (y_g, m_g, s_g) = gpu_exec(nnc, fwd, None, 0, fin, mk())
    assert st_r == 0 and st_g == 0
    assert_close(y_g, y_r, 1e-4, "y"), assert_close(m_g, m_r, 1e-5, "mean"), assert_close(s_g, s_r, 1e-4, "inv_std")
    g = seeded(shape, 4, -1, 1)
    bwd = _gnorm(abi.CCV_NNC_GROUP_NORM_BACKWARD, group_axis, groups, 1e-5, affine, reduce_axes)
    if affine:
        ins = [g, None, None, x, scale, None, None, m_r, s_r]
        mk = lambda: [np.zeros(shape, np.float32), np.zeros(pshape, np.float32), np.zeros(pshape, np.float32)]
    else:
        ins = [g, None, None, x, None, m_r, s_r]
        mk = lambda: [np.zeros(shape, np.float32)]
    st_r, outs_r = ref_exec(ref, bwd, None, 0, ins, mk())
    ins_g = [m_g if a is m_r else s_g if a is s_r else a for a in ins]  # each side's own saved statistics (compared above)
    st_g, outs_g = gpu_exec(nnc, bwd, None, 0, ins_g, mk())
    assert st_r == 0 and st_g == 0
    for name, a, b in zip(("dx", "dscale", "dbias"), outs_g, outs_r):
        assert_close(a, b, 1e-3, name)


@pytest.mark.parametrize("shape,axes", [((6, 10, 64), (2,)), ((4, 3, 5, 40), (1, 2, 3))])
def test_rmsnorm_forward_backward(gpu, ref, shape, axes):
    nnc = gpu
    x = seeded(shape, 1, -1, 1)
    rshape = tuple(1 if i in axes else d for i, d in enumerate(shape))
    pshape = tuple(d if i in axes else 1 for i, d in enumerate(shape))
    scale = seeded(pshape, 2)
    fwd = _rms(abi.CCV_NNC_RMSNORM_FORWARD, 1e-5, axes)
    mk = lambda: [np.zeros(shape, np.float32), np.zeros(rshape, np.float32)]
    st_r, (y_r, s_r) = ref_exec(ref, fwd, None, 0, [x, scale], mk())
    st_g, (y_g, s_g) = gpu_exec(nnc, fwd, None, 0, [x, scale], mk())
    assert st_r == 0 and st_g == 0
    assert_close(y_g, y_r, 1e-4, "y"), assert_close(s_g, s_r, 1e-4, "inv_std")
    g = seeded(shape, 4, -1, 1)
    bwd = _rms(abi.CCV_NNC_RMSNORM_BACKWARD, 1e-5, axes)
    ins = [g, None, x, scale, None, s_r]
    mk = lambda: [np.zeros(shape, np.float32), np.zeros(pshape, np.float32)]
    st_r, (h_r, ds_r) = ref_exec(ref, bwd, None, 0, ins, mk())
    st_g, (h_g, ds_g) = gpu_exec(nnc, bwd, None, 0, ins, mk())
    assert st_r == 0 and st_g == 0
    assert_close(h_g, h_r, 1e-3, "dx"), assert_close(ds_g, ds_r, 1e-3, "dscale")


@pytest.mark.parametrize("fmt", [NHWC, NCHW])
@pytest.mark.parametrize("kind", [abi.CCV_NNC_UPSAMPLE_NEAREST, abi.CCV_NNC_UPSAMPLE_BILINEAR])
@pytest.mark.parametrize("align", [0, 1])
def test_upsample_forward_backward(gpu, ref, fmt, kind, align):
    """test/unit/nnc/upsample.tests.c / test/int/nnc/upsample.tests.c: 2x (and a non-integer 1.5x) in both layouts."""
    nnc = gpu
    for (H, W, OH, OW) in ((7, 5, 14, 10), (6, 8, 9, 12)):
        ishape = (2, H, W, 3) if fmt == NHWC else (2, 3, H, W)
        oshape = (2, OH, OW, 3) if fmt == NHWC else (2, 3, OH, OW)
        a = seeded(ishape, 1, -1, 1)

        def mk(cmd_id):
            c = _nnc._simple(cmd_id, (2, 2, 1))
            u = c.info.upsample
            u.type, u.width_scale, u.height_scale, u.align_corners = kind, OW / W, OH / H, align
            return c
        st_r, (b_r,) = ref_exec(ref, mk(abi.CCV_NNC_UPSAMPLE_FORWARD), None, 0, [a], [np.zeros(oshape, np.float32)], fmt=fmt)
        st_g, (b_g,) = gpu_exec(nnc, mk(abi.CCV_NNC_UPSAMPLE_FORWARD), None, 0, [a], [np.zeros(oshape, np.float32)], fmt=fmt)
        assert st_r == 0 and st_g == 0
        assert_close(b_g, b_r, 1e-6, "upsample forward")
        g = seeded(oshape, 2, -1, 1)
        st_r, (h_r,) = ref_exec(ref, mk(abi.CCV_NNC_UPSAMPLE_BACKWARD), None, 0, [g], [np.zeros(ishape, np.float32)], fmt=fmt)
        st_g, (h_g,) = gpu_exec(nnc, mk(abi.CCV_NNC_UPSAMPLE_BACKWARD), None, 0, [g], [np.zeros(ishape, np.float32)], fmt=fmt)
        assert st_r == 0 and st_g == 0
        assert_close(h_g, h_r, 1e-5, "upsample backward")
