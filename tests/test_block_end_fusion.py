"""Graph rewrites (h) and (i) of ccv_nnc_sm100_graph_fuse: the end of a residual block.

(h) BATCH_NORM_FORWARD (no ReLU) ; EWSUM + RELU_FORWARD (fused add + ReLU) on its output: the batch norm only computes the
    statistics and its coefficients, the add node computes relu(x * a + b + shortcut) from the batch norm's input.
(i) EWSUM + RELU_BACKWARD (or a plain RELU_BACKWARD) ; BATCH_NORM_BACKWARD of its output: the first node also produces the batch
    norm's reduction over the gradient it writes.

Both are built to give the same bits as the unfused pair, so every case runs the same graph with CCV_NNC_SM100_FUSE_BLOCK_END=0
and without it and asks for np.array_equal on every output."""
import os

import numpy as np
import pytest

from ccv_b200 import abi, resnet50
from tests.util import pack16, seeded

pytestmark = pytest.mark.gpu
ENV = "CCV_NNC_SM100_FUSE_BLOCK_END"
DTYPES = {"f32": abi.CCV_32F, "bf16": abi.CCV_16BF, "f16": abi.CCV_16F}


def _fuse(g, block_end):
    old = os.environ.get(ENV)
    os.environ[ENV] = "1" if block_end else "0"
    try:
        return g.fuse()
    finally:
        if old is None:
            del os.environ[ENV]
        else:
            os.environ[ENV] = old


class _Tensors(object):
    """GPU tensors of one run, freed together"""

    def __init__(self, nnc):
        self.nnc, self.all = nnc, []

    def new(self, shape, dt=abi.CCV_32F, value=None):
        t = self.nnc.gpu_tensor(list(shape), datatype=dt)
        self.all.append(t)
        if value is not None:
            t.upload(value if dt == abi.CCV_32F else pack16(value, dt))
        return t

    def free(self):
        for t in self.all:
            t.free()


def _forward(nnc, dt, C, algo, block_end, bn_relu=False, y_read_later=False):
    """conv -> BN -> EWSUM(y, shortcut) -> RELU in place; returns (kinds, node inputs / outputs counts, downloaded outputs)"""
    N, H, Cin = 2, 7, 32
    ts = _Tensors(nnc)
    stream = nnc.Stream(0)
    x = ts.new((N, H, H, Cin), dt, seeded((N, H, H, Cin), 1, -1, 1))
    w = ts.new((C, 1, 1, Cin), dt, seeded((C, 1, 1, Cin), 2, -1, 1) / Cin ** 0.5)
    short = ts.new((N, H, H, C), dt, seeded((N, H, H, C), 3, -1, 1))
    scale, bias = ts.new((1, 1, 1, C), value=seeded((1, 1, 1, C), 4, 0.5, 1.5)), ts.new((1, 1, 1, C), value=seeded((1, 1, 1, C), 5, -1, 1))
    mean, var = ts.new((1, 1, 1, C), value=np.zeros((1, 1, 1, C), np.float32)), ts.new((1, 1, 1, C), value=np.ones((1, 1, 1, C), np.float32))
    sm, sis = ts.new((1, 1, 1, C)), ts.new((1, 1, 1, C))
    y, out, later = ts.new((N, H, H, C), dt), ts.new((N, H, H, C), dt), ts.new((N, H, H, C), dt)
    g = nnc.Graph()
    g.exec_new(nnc.CMD_CONVOLUTION_FORWARD(1, C, 1, 1, Cin, algorithm=algo), nnc.hint((1, 1), (0, 0)), 0, [x, w], [y])
    z = ts.new((N, H, H, C), dt)
    g.exec_new(nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9), None, 0, [y, scale, bias, mean, var], [z, mean, var, sm, sis])
    if bn_relu:
        g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [z], [z])
    g.exec_new(nnc.CMD_EWSUM_FORWARD(), None, 0, [z, short], [out])
    g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [out], [out])
    if y_read_later:
        g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [z], [later])
    n_before = len(g)
    removed = _fuse(g, block_end)
    assert len(g) == n_before - removed
    nodes = g.nodes()
    assert g.run(stream) == 0
    stream.wait()
    res = dict(out=out.download(), mean=mean.download(), var=var.download(), sm=sm.download(), sis=sis.download(), conv=y.download())
    if y_read_later:
        res["later"] = later.download()
    ts.free(), g.free(), stream.free()
    return nodes, removed, res


def _same(a, b, what):
    for k in a:
        assert np.array_equal(a[k], b[k]), "%s: %s differs with the block-end rewrites on" % (what, k)


@pytest.mark.parametrize("dtype", sorted(DTYPES))
@pytest.mark.parametrize("C", [64, 256, 2048])
@pytest.mark.parametrize("algo", [abi.CCV_NNC_SM100_ALGO_TF32, abi.CCV_NNC_SM100_ALGO_FFMA])
def test_forward_bn_add_relu_is_bit_identical(gpu, dtype, C, algo):
    nnc = gpu
    if algo == abi.CCV_NNC_SM100_ALGO_FFMA and dtype != "f32":
        pytest.skip("the CUDA-core convolution is fp32")
    dt = DTYPES[dtype]
    on_nodes, on_removed, on = _forward(nnc, dt, C, algo, True)
    off_nodes, off_removed, off = _forward(nnc, dt, C, algo, False)
    assert on_removed == off_removed
    kinds = [k for _, k, _, _ in on_nodes]
    assert kinds == [6 if algo != abi.CCV_NNC_SM100_ALGO_FFMA else 0, 7, 3], kinds
    # statistics-only batch norm: the coefficient tensor is a 6th output; the add reads x, the shortcut and the coefficients
    assert len(on_nodes[1][3]) == 6 and len(off_nodes[1][3]) == 5
    assert len(on_nodes[2][2]) == 3 and on_nodes[2][2][0] == on_nodes[0][3][0] and len(off_nodes[2][2]) == 2
    _same(on, off, "forward %s C=%d algo=%d" % (dtype, C, algo))


def test_forward_not_rewritten_when_the_bn_output_is_read_later(gpu):
    nnc = gpu
    nodes, _, on = _forward(nnc, abi.CCV_32F, 64, abi.CCV_NNC_SM100_ALGO_TF32, True, y_read_later=True)
    _, _, off = _forward(nnc, abi.CCV_32F, 64, abi.CCV_NNC_SM100_ALGO_TF32, False, y_read_later=True)
    assert len(nodes[1][3]) == 5 and len(nodes[2][2]) == 2, [(k, len(i), len(o)) for _, k, i, o in nodes]
    _same(on, off, "forward, y read later")


def test_forward_not_rewritten_when_the_bn_has_a_relu(gpu):
    nnc = gpu
    nodes, _, on = _forward(nnc, abi.CCV_32F, 64, abi.CCV_NNC_SM100_ALGO_TF32, True, bn_relu=True)
    _, _, off = _forward(nnc, abi.CCV_32F, 64, abi.CCV_NNC_SM100_ALGO_TF32, False, bn_relu=True)
    assert [k for _, k, _, _ in nodes] == [6, 1, 3]
    assert len(nodes[1][3]) == 5 and len(nodes[2][2]) == 2
    _same(on, off, "forward, bn + relu")


def _backward(nnc, dt, C, with_add, block_end):
    """[EWSUM(ga, gb -> ga) ;] RELU_BACKWARD(ga, mask yb) -> BN_BACKWARD -> CONVOLUTION_BACKWARD with a bias gradient"""
    N, H, Cin = 4, 7, 32
    ts = _Tensors(nnc)
    stream = nnc.Stream(0)
    rs = np.random.RandomState(5)
    ga = ts.new((N, H, H, C), dt, rs.randn(N, H, H, C).astype(np.float32))
    gb = ts.new((N, H, H, C), dt, rs.randn(N, H, H, C).astype(np.float32))
    yb = ts.new((N, H, H, C), dt, rs.randn(N, H, H, C).astype(np.float32))  # the block output: the ReLU mask
    xv = rs.randn(N, H, H, C).astype(np.float32) * 2 + 0.5
    x = ts.new((N, H, H, C), dt, xv)
    xin = ts.new((N, H, H, Cin), dt, seeded((N, H, H, Cin), 1, -1, 1))
    w = ts.new((C, 1, 1, Cin), dt, seeded((C, 1, 1, Cin), 2, -1, 1) / Cin ** 0.5)
    scale = ts.new((1, 1, 1, C), value=seeded((1, 1, 1, C), 4, 0.5, 1.5))
    mean = ts.new((1, 1, 1, C), value=xv.mean(axis=(0, 1, 2)).reshape(1, 1, 1, C).astype(np.float32))
    istd = ts.new((1, 1, 1, C), value=(1.0 / np.sqrt(xv.var(axis=(0, 1, 2)) + 1e-4)).reshape(1, 1, 1, C).astype(np.float32))
    dx, h = ts.new((N, H, H, C), dt), ts.new((N, H, H, Cin), dt)
    dscale, dbias = ts.new((1, 1, 1, C)), ts.new((1, 1, 1, C))
    dw, cdb = ts.new((C, 1, 1, Cin), dt), ts.new((C,), dt)
    g = nnc.Graph()
    if with_add:
        g.exec_new(nnc.CMD_EWSUM_FORWARD(), None, 0, [ga, gb], [ga])
    g.exec_new(nnc.CMD_RELU_BACKWARD(), None, 0, [ga, None, yb], [ga])
    g.exec_new(nnc.CMD_BATCH_NORM_BACKWARD(1e-4, 0, 0.9), None, 0, [ga] + [None] * 4 + [x, scale] + [None] * 6 + [mean, istd], [dx, dscale, dbias])
    g.exec_new(nnc.CMD_CONVOLUTION_BACKWARD(1, C, 1, 1, Cin), nnc.hint((1, 1), (0, 0)), 0, [dx, xin, w], [h, dw, cdb])
    removed = _fuse(g, block_end)
    nodes = g.nodes()
    assert g.run(stream) == 0
    stream.wait()
    res = dict(g=ga.download(), dx=dx.download(), dscale=dscale.download(), dbias=dbias.download(), cdb=cdb.download(), dw=dw.download(), h=h.download())
    ts.free(), g.free(), stream.free()
    return nodes, removed, res


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("C", [64, 256, 2048])
@pytest.mark.parametrize("with_add", [True, False])
def test_backward_add_relu_carries_the_bn_reduction_bit_identically(gpu, dtype, C, with_add):
    nnc = gpu
    dt = DTYPES[dtype]
    on_nodes, on_removed, on = _backward(nnc, dt, C, with_add, True)
    off_nodes, off_removed, off = _backward(nnc, dt, C, with_add, False)
    assert on_removed == off_removed
    kinds = [k for _, k, _, _ in on_nodes]
    assert kinds == [4, 8, 0], kinds
    # the add / ReLU backward node also takes x and the saved mean and writes the partial rows the batch norm reads as a 16th input
    assert len(on_nodes[0][2]) == 5 and len(on_nodes[0][3]) == 2 and len(on_nodes[1][2]) == 16
    assert on_nodes[1][2][15] == on_nodes[0][3][1]
    assert [k for _, k, _, _ in off_nodes] == [4 if with_add else 0, 8, 0] and len(off_nodes[1][2]) == 15
    _same(on, off, "backward %s C=%d add=%s" % (dtype, C, with_add))


@pytest.mark.parametrize("dtype,algo", [(abi.CCV_32F, abi.CCV_NNC_SM100_ALGO_TF32), (abi.CCV_16BF, -1)])
def test_whole_resnet50_is_bit_identical(gpu, dtype, algo):
    nnc = gpu
    rs = np.random.RandomState(0)
    x, lab = rs.rand(4, 64, 64, 3).astype(np.float32), (np.arange(4) % 10).astype(np.int32)

    def run(block_end):
        stream = nnc.Stream(0)
        net = resnet50.Net(4, image=64, classes=10, seed=7, algorithm=algo, dtype=dtype)
        net.input.upload(x if dtype == abi.CCV_32F else pack16(x, dtype)), net.labels.upload(lab)
        g = nnc.Graph()
        for cmd, hint, flags, ins, outs in net.fwd + net.bwd:
            g.exec_new(cmd, hint, flags, ins, outs)
        _fuse(g, block_end)
        kinds = [k for _, k, _, _ in g.nodes()]
        assert g.run(stream) == 0
        stream.wait()
        res = dict(logits=net.logits.download(), loss=net.loss.download(), g_flat=net.g_flat.download())
        if getattr(net, "g_flat_b", None) is not None:
            res["g_flat_b"] = net.g_flat_b.download()
        g.free(), net.free(), stream.free()
        return kinds, res

    k_on, on = run(True)
    k_off, off = run(False)
    # same node list; the one plain RELU_BACKWARD (the last block's, whose mask is the block output) becomes a kind-4 node
    assert len(k_on) == len(k_off) and k_on.count(4) == k_off.count(4) + 1
    _same(on, off, "resnet50")
