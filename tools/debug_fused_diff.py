"""GPU debug: where do the fused and the unfused ResNet-50 graphs (tests/test_resnet_parity.py configuration) first differ?
Prints, layer by layer, the normalised max difference of every activation and of the batch-norm saved statistics."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ccv_b200 import nnc, resnet50

BATCH, IMAGE, CLASSES = 4, 96, 10
algo = int(sys.argv[1]) if len(sys.argv) > 1 else -1
nnc.init()
stream = nnc.Stream(0)
rs = np.random.RandomState(0)
x, lab = rs.rand(BATCH, IMAGE, IMAGE, 3).astype(np.float32), (np.arange(BATCH) % CLASSES).astype(np.int32)


def build(fuse):
    """the net after one step, and the data pointers of the activations its graph writes"""
    net = resnet50.Net(BATCH, image=IMAGE, classes=CLASSES, seed=7, algorithm=algo)
    net.input.upload(x), net.labels.upload(lab)
    g = nnc.Graph()
    for n in net.fwd + net.bwd:
        g.exec_new(*n)
    if fuse:
        g.fuse()
    assert g.run(stream) == 0
    stream.wait()
    # a statistics-only batch norm (rewrite (h): 6 outputs, the last one its coefficients) keeps y in its output list but does
    # not write it: the residual add behind it reads the batch norm's input instead
    written = set()
    for _, kind, _, outs in g.nodes():
        written.update(o for o in (outs[1:] if kind == 7 and len(outs) == 6 else outs) if o)
    return net, written


def err(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


(plain, _), (fused, fused_written) = build(False), build(True)
for lp, lf in zip(plain.layers, fused.layers):
    k = lp["kind"]
    line = "%-28s %-9s" % (lp["name"], k)
    if "y" in lp and lp["y"] is not None:
        line += " y %.2e" % err(lf["y"].download(), lp["y"].download()) if lf["y"].ptr in fused_written else " y (not written by the fused graph)"
    if k == "bn":
        sis = lp["sis"].download()
        line += " mean %.2e inv_std %.2e (max inv_std %.1f)" % (err(lf["sm"].download(), lp["sm"].download()), err(lf["sis"].download(), sis), float(sis.max()))
    print(line)
print("logits", err(fused.logits.download(), plain.logits.download()))
