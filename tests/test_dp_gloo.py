"""The N>1 path on CPU: two gloo ranks, each running its batch shard of a small command-list model on the oracle
(CCV_NNC_BACKEND_CPU_REF), one sum-allreduce of the flat gradient buffer (ccv_b200/dp.py), then the SGD commands, must
reproduce the single-process result on the concatenated batch -- the check of test/int/nnc/parallel.tests.c:192-371
(2-way data parallel vs one device), minus the GPUs."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r"""
import os, sys
import numpy as np
sys.path.insert(0, %(root)r)
import torch.distributed as dist
from ccv_b200 import dp, resnet50
from oracle import ref_factory


class TinyNet(resnet50.Net):
    # conv 3x3/2 -> relu -> conv 3x3 -> relu -> flatten -> dense -> softmax -> CCE; no batch norm (its statistics are
    # per replica by design) and no pooling (CPU_REF only walks image 0)
    def _build_body(self, x, xs):
        x, xs = self._conv(x, xs, 3, 8, 3, 2, 1, True, "c0", need_dx=False)
        x = self._relu(x, xs, "r0")
        x, xs = self._conv(x, xs, 8, 8, 3, 1, 1, True, "c1")
        x = self._relu(x, xs, "r1")
        return x, xs


def run(batch, global_batch, x, y):
    net = TinyNet(batch, image=8, classes=5, global_batch=global_batch, factory=ref_factory.RefFactory(), seed=3, learn_rate=0.1)
    net.input.upload(x), net.labels.upload(y)
    ref_factory.run_nodes(net.fwd), ref_factory.run_nodes(net.bwd)
    return net


rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
rs = np.random.RandomState(0)
X, Y = rs.rand(4, 8, 8, 3).astype(np.float32), rs.randint(0, 5, size=(4,)).astype(np.int32)
net = run(4 // world, 4, dp.shard(X, rank, world), dp.shard(Y, rank, world))
dp.FlatAllreduce(net, dist)()
ref_factory.run_nodes(net.opt)
if rank == 0:
    full = run(4, 4, X, Y)
    ref_factory.run_nodes(full.opt)
    a, b = net.w_flat.download(), full.w_flat.download()
    err = float(np.abs(a - b).max() / np.abs(b).max())
    g = float(np.abs(net.g_flat.download() - full.g_flat.download()).max() / np.abs(full.g_flat.download()).max())
    print("DP_RESULT weights_err=%%.3e grads_err=%%.3e changed=%%d" %% (err, g, int(np.abs(full.w_flat.download() - full.param_host).max() > 0)))
dist.barrier()
dist.destroy_process_group()
"""


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.ref
def test_two_rank_data_parallel_matches_single_process(ref, tmp_path):
    if getattr(ref, "stored", False):
        pytest.skip("the ranks run the model on the compiled reference (oracle/_ref/libccv_ref.so, make -C oracle)")
    script = tmp_path / "dp_worker.py"
    script.write_text(WORKER % dict(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(_free_port()), WORLD_SIZE="2", OMP_NUM_THREADS="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=300)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    line = [l for l in outs[0].splitlines() if l.startswith("DP_RESULT")][0]
    vals = dict(kv.split("=") for kv in line.split()[1:])
    assert float(vals["grads_err"]) < 1e-5 and float(vals["weights_err"]) < 1e-6 and vals["changed"] == "1", line
