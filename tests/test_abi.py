"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/ccv_nnc_sm100.h
declares, and its struct layouts / identifiers match the reference's own headers (through oracle/_ref)."""
import ctypes as C
import hashlib
import json
import os
import re

import pytest

from ccv_b200 import abi, nnc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "ccv_nnc_sm100.h")).read()
    cmds = re.search(r"#define CCV_NNC_SM100_COMMANDS\(X\)(.*?)\n\n", text, re.S).group(1)
    names = re.findall(r"X\((\w+)\)", cmds)
    syms = ["_register_command_%s_backend_CCV_NNC_BACKEND_GPU_SM100" % n for n in names]
    # plain function declarations: "type name(args);" at the start of a line
    for m in re.finditer(r"^(?:[\w\*]+\s+)+\**(ccv_nnc_\w+)\s*\(", text, re.M):
        syms.append(m.group(1))
    return sorted(set(syms)), names


def test_library_exports_every_declared_symbol():
    lib = nnc.lib()
    syms, names = _declared_symbols()
    assert len(names) >= 40
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, "symbols declared in include/ccv_nnc_sm100.h but not exported: %s" % missing


def test_registration_fills_registry_records():
    class Registry(C.Structure):
        _fields_ = [("tensor_formats", C.c_int), ("tensor_datatypes", C.c_int), ("tensor_memory", C.c_int), ("algorithms", C.c_int),
                    ("exec", C.c_void_p), ("autotune", C.c_void_p), ("aux", C.c_void_p)]
    lib = nnc.lib()
    _, names = _declared_symbols()
    for n in names:
        r = Registry()
        getattr(lib, "_register_command_%s_backend_CCV_NNC_BACKEND_GPU_SM100" % n)(C.byref(r))
        assert r.exec, n
        assert r.tensor_memory & abi.CCV_TENSOR_GPU_MEMORY, n
        assert r.tensor_formats and r.tensor_datatypes and r.algorithms >= 1, n


def test_backend_and_command_ids_follow_the_generator_rule():
    # lib/nnc/cmd/build-cmd.rb:292,386: id = first 4 bytes of SHA256(name), commands with the low bit cleared
    def h(name):
        return int.from_bytes(hashlib.sha256(name.encode()).digest()[:4], "big")
    assert h("CCV_NNC_BACKEND_GPU_SM100") == abi.CCV_NNC_BACKEND_GPU_SM100
    assert h("CCV_NNC_BACKEND_CPU_REF") == abi.CCV_NNC_BACKEND_CPU_REF
    for name, val in abi.CMD_IDS.items():
        assert h("CCV_NNC_%s" % name) & ~1 == val, name  # hashed without the _FORWARD/_BACKWARD suffix (build-cmd.rb:276-283)


def test_dispatch_finds_the_backend_and_refuses_cpu_tensors():
    nnc.init()
    assert nnc.lib().ccv_nnc_cmd_ok(abi.CCV_NNC_GEMM_FORWARD, abi.CCV_NNC_BACKEND_GPU_SM100) == 1
    assert nnc.lib().ccv_nnc_cmd_ok(abi.CCV_NNC_GEMM_FORWARD, abi.CCV_NNC_BACKEND_CPU_REF) == 0
    # no CPU fallback: a command on host tensors with no backend named has no kernel
    import numpy as np
    a, b, c = nnc.cpu_tensor([2, 2]), nnc.cpu_tensor([2, 2]), nnc.cpu_tensor([2, 2])
    a.upload(np.eye(2)), b.upload(np.eye(2))
    cmd = nnc.CMD_GEMM_FORWARD(backend=0)
    assert nnc.cmd_exec(cmd, None, 0, [a, b], [c]) == abi.CCV_NNC_EXEC_NO_KERNEL
    for t in (a, b, c):
        t.free()


@pytest.mark.ref
def test_struct_layouts_match_the_reference_headers(ref):
    if getattr(ref, "stored", False):  # what the compiled reference reported (tests/golden/make_golden.py)
        out = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_facts.json")))["abi_sizes"]
    else:
        out = (C.c_int * 10)()
        ref.ref().ref_abi_sizes(out)
    assert list(out)[:6] == [C.sizeof(abi.Cmd), C.sizeof(abi.Hint), C.sizeof(abi.CmdParam), C.sizeof(abi.TensorParam), C.sizeof(abi.Tensor), C.sizeof(abi.TensorView)]
    assert out[6] == abi.Cmd.info.offset and out[7] == abi.Tensor.info.offset and out[8] == abi.TensorView.stride.offset and out[9] == abi.Tensor.data.offset


def test_tensor_views_carry_offset_and_strides():
    import numpy as np
    t = nnc.cpu_tensor([4, 6])
    t.upload(np.arange(24).reshape(4, 6))
    v = nnc.tensor_view_new(t, [2, 3], [1, 2, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0], [6, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0])
    s = v.struct
    assert s.type & abi.CCV_TENSOR_VIEW
    assert s.data - t.struct.data == (1 * 6 + 2) * 4
    assert list(s.stride)[:2] == [6, 1] and s.contiguous == 0
    v.free(), t.free()
