"""Host logic of the flat graph (ccv_b200/csrc/nnc_host.cu), on CPU: ccv_nnc_sm100_graph_fuse only inspects node descriptions
and tensor identities, so its rewrites can be checked without a device (nothing is executed here; tensors are host tensors).
Rewrite (f) (convolution -> batch-norm statistics) needs a device allocation and is covered by the GPU tests."""
import ctypes as C

import pytest

from ccv_b200 import abi, nnc


def _t(*dims):
    return nnc.cpu_tensor(list(dims))


def _bn_back_inputs(g, x, scale, mean, istd):
    return [g] + [None] * 4 + [x, scale] + [None] * 6 + [mean, istd]


def test_fuse_rewrites_pairs_runs_and_links():
    nnc.init()
    N, H, C, K = 2, 4, 8, 16
    x, w, b, y, z = _t(N, H, H, C), _t(K, 3, 3, C), _t(K), _t(N, H, H, K), _t(N, H, H, K)
    scale, bias, mean, var, sm, sis = (_t(1, 1, 1, K) for _ in range(6))
    short, out = _t(N, H, H, K), _t(N, H, H, K)
    g = nnc.Graph()
    hint = nnc.hint((1, 1), (1, 1))
    # forward: conv -> bn -> relu (in place) -> ewsum(z, short) -> relu (in place)
    g.exec_new(nnc.CMD_CONVOLUTION_FORWARD(1, K, 3, 3, C), hint, 0, [x, w, b], [y])
    g.exec_new(nnc.CMD_BATCH_NORM_FORWARD(1e-4, 0, 0.9), None, 0, [y, scale, bias, mean, var], [z, mean, var, sm, sis])
    g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [z], [z])
    g.exec_new(nnc.CMD_EWSUM_FORWARD(), None, 0, [z, short], [out])
    g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [out], [out])
    # backward: relu_bwd (in place on gz, mask z) -> bn_bwd -> conv_bwd with a bias gradient
    gz, gy, gx, dw, db, dscale, dbias = _t(N, H, H, K), _t(N, H, H, K), _t(N, H, H, C), _t(K, 3, 3, C), _t(K), _t(1, 1, 1, K), _t(1, 1, 1, K)
    g.exec_new(nnc.CMD_RELU_BACKWARD(), None, 0, [gz, None, z], [gz])
    g.exec_new(nnc.CMD_BATCH_NORM_BACKWARD(1e-4, 0, 0.9), None, 0, _bn_back_inputs(gz, y, scale, sm, sis), [gy, dscale, dbias])
    g.exec_new(nnc.CMD_CONVOLUTION_BACKWARD(1, K, 3, 3, C), hint, 0, [gy, x, w], [gx, dw, db])
    # optimizer: two hyper-parameter groups, interleaved (weights with decay, biases / norm parameters without)
    params = [(_t(64), _t(64), _t(64)) for _ in range(6)]
    for i, (gr, a, m) in enumerate(params):
        decay = 1e-4 if i % 2 == 0 else 0.0
        g.exec_new(nnc.CMD_SGD_FORWARD(1, 0.1, 1.0 / 256, decay, 0.9, 0.0), None, 0, [gr, a, m], [a, m])
    n_before = len(g)
    removed = g.fuse()
    nodes = g.nodes()
    kinds = [k for _, k, _, _ in nodes]
    cmds = [c for c, _, _, _ in nodes]
    # bn+relu (1), add+relu (3), relu_bwd+bn_bwd (2), two multi-tensor SGD nodes (5); the convolutions stay plain on host tensors
    assert kinds == [0, 1, 3, 2, 0, 5, 5], kinds
    assert cmds[0] == abi.CCV_NNC_CONVOLUTION_FORWARD and cmds[4] == abi.CCV_NNC_CONVOLUTION_BACKWARD
    assert removed == n_before - len(nodes) == 3 + 4
    # (b): the fused relu+bn backward carries the forward bias in input slot 7 ...
    _, _, ins, outs = nodes[3]
    assert len(ins) == 15 and ins[7] == bias.ptr and ins[0] == gz.ptr
    # ... and (g): it also writes the convolution's bias gradient (4th output); the convolution no longer asks for it
    assert len(outs) == 4 and outs[3] == db.ptr
    _, _, cins, couts = nodes[4]
    assert couts[2] is None and couts[0] == gx.ptr and couts[1] == dw.ptr
    # (e): SGD nodes grouped by hyper-parameters, three (g, a, m) triples each, in their original relative order
    for node, group in ((nodes[5], params[0::2]), (nodes[6], params[1::2])):
        _, _, sins, souts = node
        assert sins == [t.ptr for triple in group for t in triple]
        assert souts == [t.ptr for (_, a, m) in group for t in (a, m)]
    g.free()


def test_fuse_leaves_unrelated_and_dependent_nodes_alone():
    nnc.init()
    a, b, c = _t(32), _t(32), _t(32)
    g = nnc.Graph()
    # relu whose input is not the batch norm's output; ewsum followed by a relu on a different tensor
    g.exec_new(nnc.CMD_EWSUM_FORWARD(), None, 0, [a, b], [c])
    g.exec_new(nnc.CMD_RELU_FORWARD(), None, 0, [a], [a])
    # two SGD nodes where the second reads what the first writes: must stay separate
    m1, m2, g1 = _t(32), _t(32), _t(32)
    g.exec_new(nnc.CMD_SGD_FORWARD(0, 0.1, 1.0, 0.0, 0.9, 0.9), None, 0, [g1, a, m1], [b, m1])
    g.exec_new(nnc.CMD_SGD_FORWARD(0, 0.1, 1.0, 0.0, 0.9, 0.9), None, 0, [g1, b, m2], [c, m2])
    assert g.fuse() == 0
    assert [k for _, k, _, _ in g.nodes()] == [0, 0, 0, 0]
    g.free()


def test_comm_plumbing_without_a_device():
    """The communicator side channel is host-only: rank 0's 128-byte id can be produced without a GPU (NCCL is dlopen'ed), and the
    allreduce command refuses host tensors instead of touching them (no CPU fallback)."""
    nnc.init()
    try:
        a, b = nnc.comm_unique_id(), nnc.comm_unique_id()
    except RuntimeError:
        import pytest
        pytest.skip("libnccl.so.2 not loadable here")
    assert len(a) == 128 and len(b) == 128 and a != b
    x = _t(16)
    assert nnc.cmd_exec(nnc.CMD_COMM_ALLREDUCE_FORWARD(), None, 0, [x], [x]) != 0


def test_gradient_buckets_cover_the_flat_buffer_and_follow_their_producers():
    """ccv_b200/resnet50.py backward_with_exchange (host logic, oracle-side tensors): the allreduce nodes partition the flat
    gradient buffer, and each sits behind the last backward node that writes into its bucket."""
    from oracle import ref, ref_factory
    if not ref.available():
        pytest.skip("oracle/_ref/libccv_ref.so not built")
    from ccv_b200 import abi, resnet50
    net = resnet50.Net(2, image=32, classes=10, factory=ref_factory.RefFactory())
    nodes, side = net.backward_with_exchange(4)
    assert len(side) == 4 and len(nodes) == len(net.bwd) + 4
    base = net.g_flat.array.ctypes.data
    spans = []
    for i in side:
        cmd, _, _, ins, outs = nodes[i]
        assert cmd.cmd == abi.CCV_NNC_COMM_ALLREDUCE_FORWARD and ins == outs
        assert nodes[i - 1][0].cmd in (abi.CCV_NNC_CONVOLUTION_BACKWARD, abi.CCV_NNC_GEMM_BACKWARD) or i == len(nodes) - 1
        lo = (ins[0].array.ctypes.data - base) // 4
        spans.append((lo, lo + ins[0].array.size, i))
    spans.sort()
    assert spans[0][0] == 0 and spans[-1][1] == net.flat_count and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    # every gradient tensor of a bucket is written by a node in front of the bucket's allreduce
    for lo, hi, at in spans:
        for j in range(at + 1, len(nodes)):
            for t in nodes[j][4]:
                if t is not None and hasattr(t, "array") and nodes[j][0].cmd != abi.CCV_NNC_COMM_ALLREDUCE_FORWARD:
                    off = (t.array.ctypes.data - base) // 4
                    assert not (0 <= off < net.flat_count and lo <= off < hi), "a gradient of bucket [%d, %d) is written after its allreduce" % (lo, hi)
