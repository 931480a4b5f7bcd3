"""Shared helpers for the parity tests: run one command on the SM100 backend (through the C ABI) and on the oracle
(the reference's own CCV_NNC_BACKEND_CPU_REF) from the same numpy inputs."""
import atexit
import hashlib
import json
import os
import struct

import numpy as np

from ccv_b200 import abi

NHWC = abi.CCV_TENSOR_FORMAT_NHWC
NCHW = abi.CCV_TENSOR_FORMAT_NCHW
NP_TO_CCV = {np.dtype(np.float32): abi.CCV_32F, np.dtype(np.int32): abi.CCV_32S, np.dtype(np.float64): abi.CCV_64F, np.dtype(np.float16): abi.CCV_16F, np.dtype(np.uint16): abi.CCV_16F, np.dtype(np.uint8): abi.CCV_8U}


def seeded(shape, seed, lo=0.0, hi=1.0, dtype=np.float32):
    """U(lo, hi] inputs, seeded (the reference's GPU-vs-CPU protocol, test/int/nnc/cudnn.tests.c:38-46, uses dSFMT seed 0)."""
    r = np.random.RandomState(seed)
    return (lo + (hi - lo) * (1.0 - r.random_sample(shape))).astype(dtype)


def gpu_exec(nnc, cmd, hint, flags, in_arrays, out_arrays, fmt=NHWC, in_fmts=None, out_fmts=None, stream=None):
    """Upload, ccv_nnc_cmd_exec on CCV_NNC_BACKEND_GPU_SM100, download. The same array object appearing in both lists
    (or twice) is the same GPU tensor (in-place ops). Returns (status, [output arrays])."""
    cache = {}

    def tensor_for(a, f):
        if a is None:
            return None
        if id(a) not in cache:
            t = nnc.gpu_tensor(list(a.shape), f, NP_TO_CCV[a.dtype])
            t.upload(a.view(np.float16) if a.dtype == np.uint16 else a)
            cache[id(a)] = t
        return cache[id(a)]

    ins = [tensor_for(a, in_fmts[i] if in_fmts else fmt) for i, a in enumerate(in_arrays)]
    outs = [tensor_for(a, out_fmts[i] if out_fmts else fmt) for i, a in enumerate(out_arrays)]
    status = nnc.cmd_exec(cmd, hint, flags, ins, outs, stream)
    if stream is not None:
        stream.wait()
    results = [None if t is None else t.download() for t in outs]
    for t in cache.values():
        t.free()
    return status, results


# ---- CPU_REF outputs stored under tests/golden/cpu_ref -----------------------------------------------------------------
# Where the compiled reference (oracle/_ref/libccv_ref.so) is not built, ref_exec answers from outputs the reference computed
# for the very same call: tests/golden/cpu_ref/<test module>.npz, keyed by a digest of the command, its parameters, the hint,
# the flags and every operand's type, shape, format and bytes (the inputs are seeded, so the digest is the same on every
# machine).  An output of at most SAMPLE + 2 * EDGE + 1 elements, or one a test asks for whole, is stored whole.  A larger one is stored at
# SAMPLE seeded positions, its first and last EDGE elements and the position of its largest magnitude; the array handed to the
# test reads NaN everywhere else and is registered as sampled.  Only for a registered array (or a view of one) do the
# comparison helpers below skip NaN positions; a NaN anywhere else still fails.  Since the largest magnitude is kept, the
# normalised errors use the same denominator as on the full array.
# CCV_REF_RECORD=1 with the compiled reference present rewrites these files from it.  The outputs handed back to the test are
# then already the stored form (the reference itself still computes on whole operands), so a passing recording run is a
# passing replay.
GOLDEN_REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cpu_ref")
SAMPLE = 96
EDGE = 16
_STORE_DTYPES = {"f4": np.float32, "f8": np.float64, "f2": np.float16, "i4": np.int32, "u1": np.uint8}


class StoredRef(object):
    """Stands for the compiled reference in ref_exec when only its stored outputs are available; anything else a test asks
    of the reference skips that test."""
    stored = True

    def __getattr__(self, name):
        import pytest
        pytest.skip("needs the compiled reference (oracle/_ref/libccv_ref.so, make -C oracle): %s" % name)


def _current_module():
    test = os.environ.get("PYTEST_CURRENT_TEST", "")
    return os.path.splitext(os.path.basename(test.split("::")[0]))[0] or "none", test.split(" ")[0]


_sampled = {"test": None, "arrays": {}}   # the sampled reference outputs handed to the current test: id -> array


def _register_sampled(a):
    test = _current_module()[1]
    if test != _sampled["test"]:
        _sampled["test"], _sampled["arrays"] = test, {}
    _sampled["arrays"][id(a)] = a


def is_sampled(a):
    """True for a sampled stored reference output of the current test, or a view of one."""
    arrays = _sampled["arrays"] if _current_module()[1] == _sampled["test"] else {}
    while isinstance(a, np.ndarray):
        if arrays.get(id(a)) is a:
            return True
        a = a.base
    return False


def _call_key(cmd, hint, flags, ins, outs, fmt, in_fmts, out_fmts):
    h = hashlib.sha1(struct.pack("<Ii", cmd.cmd, flags) + bytes(cmd.info) + (bytes(hint) if hint is not None else b"-"))
    for i, a in enumerate(ins):
        h.update(b"N" if a is None else ("%s%s%d" % (a.dtype.str, a.shape, in_fmts[i] if in_fmts else fmt)).encode() + np.ascontiguousarray(a).tobytes())
    h.update(b"|")
    for i, a in enumerate(outs):
        h.update(b"N" if a is None else ("%s%s%d" % (a.dtype.str, a.shape, out_fmts[i] if out_fmts else fmt)).encode() + np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:24]


def _sample_positions(size, peak):
    picks = np.random.RandomState(size % (1 << 31)).choice(size, SAMPLE, replace=False)
    return np.unique(np.concatenate([picks, np.arange(EDGE), np.arange(size - EDGE, size), [peak]]))


def _stored_form(a, whole):
    """(array as the test sees it, stored values, peak position or -1 when stored whole)"""
    if whole or a.size <= SAMPLE + 2 * EDGE + 1 or a.dtype.kind != "f":
        return a, a.reshape(-1).copy(), -1
    flat = a.reshape(-1)
    peak = int(np.argmax(np.abs(flat.astype(np.float64))))
    pos = _sample_positions(flat.size, peak)
    seen = np.full(flat.shape, np.nan, a.dtype)
    seen[pos] = flat[pos]
    return seen.reshape(a.shape), flat[pos].copy(), peak


class _Recorder(object):
    def __init__(self):
        self.modules = {}   # module -> {key: [status, [output shape / dtype or None], [(stored values, peak) or None]]}
        self.test, self.given = None, {}   # sampled arrays handed to the current test: id -> (array, whole contents, sampled contents)

    def begin(self, test):
        if test != self.test:
            self.test, self.given = test, {}

    def restore(self, arrays):
        """Whole contents back into sampled outputs a test passes to a further reference call (the reference computes on whole
        operands; the call's key was taken on what the test holds, which is what a replay sees).  Returns what was restored."""
        done = []
        for a in arrays:
            if a is not None and id(a) in self.given and self.given[id(a)][0] is a and all(a is not d for d in done):
                a[...] = self.given[id(a)][1]
                done.append(a)
        return done

    def resample(self, arrays):
        for a in arrays:
            a[...] = self.given[id(a)][2]

    def record(self, module, key, status, outs, whole):
        entry = [status, [None if a is None else (a.dtype.str[1:], a.shape) for a in outs], []]
        for a in outs:
            if a is None:
                entry[2].append(None)
                continue
            seen, vals, peak = _stored_form(a, whole)
            entry[2].append((vals, peak))
            if peak >= 0:
                self.given[id(a)] = (a, a.copy(), seen)
                a[...] = seen
                _register_sampled(a)
            else:
                self.given.pop(id(a), None)
        self.modules.setdefault(module, {})[key] = entry

    def write(self):
        os.makedirs(GOLDEN_REF, exist_ok=True)
        for module, calls in self.modules.items():
            index, chunks = {}, {k: [] for k in _STORE_DTYPES}
            sizes = {k: 0 for k in _STORE_DTYPES}
            for key, (status, kinds, stored) in sorted(calls.items()):
                outs = []
                for k, s in zip(kinds, stored):
                    if k is None:
                        outs.append(None)
                        continue
                    code, shape = k
                    vals, peak = s
                    outs.append([code, list(shape), sizes[code], int(vals.size), peak])
                    chunks[code].append(vals)
                    sizes[code] += vals.size
                index[key] = [int(status), outs]
            arrays = {k: np.concatenate(v).astype(_STORE_DTYPES[k]) for k, v in chunks.items() if v}
            np.savez_compressed(os.path.join(GOLDEN_REF, module + ".npz"), index=np.array(json.dumps(index, sort_keys=True)), **arrays)


_recorder = None
_stored = {}


def _recording():
    global _recorder
    if _recorder is None and os.environ.get("CCV_REF_RECORD"):
        _recorder = _Recorder()
        atexit.register(_recorder.write)
    return _recorder


def _replay(module, key, out_arrays):
    if module not in _stored:
        path = os.path.join(GOLDEN_REF, module + ".npz")
        if not os.path.exists(path):
            _stored[module] = ({}, {})
        else:
            z = np.load(path)
            _stored[module] = (json.loads(str(z["index"])), {k: z[k] for k in z.files if k != "index"})
    index, values = _stored[module]
    if not index:
        import pytest
        pytest.skip("no stored CPU_REF outputs for %s (tests/golden/cpu_ref) and the compiled reference is not built" % module)
    assert key in index, "no stored CPU_REF output for this call in tests/golden/cpu_ref/%s.npz (regenerate with CCV_REF_RECORD=1 and the compiled reference)" % module
    status, outs = index[key]
    for a, o in zip(out_arrays, outs):
        if a is None or o is None:
            continue
        code, shape, off, n, peak = o
        vals = values[code][off:off + n]
        assert tuple(shape) == a.shape, (module, key, shape, a.shape)
        if peak < 0:
            a[...] = vals.reshape(a.shape)
        else:
            flat = np.full(a.size, np.nan, a.dtype)
            flat[_sample_positions(a.size, peak)] = vals
            a[...] = flat.reshape(a.shape)
            _register_sampled(a)
    return status, out_arrays


def ref_exec(ref, cmd, hint, flags, in_arrays, out_arrays, fmt=NHWC, in_fmts=None, out_fmts=None, whole=False):
    """Same command on the reference's CPU_REF. out_arrays are modified in place and returned.  With only the stored outputs
    (StoredRef), large outputs come back sampled (see above) unless `whole`: for outputs a test computes further operands from."""
    if getattr(ref, "stored", False):
        module, _ = _current_module()
        return _replay(module, _call_key(cmd, hint, flags, in_arrays, out_arrays, fmt, in_fmts, out_fmts), out_arrays)
    rec = _recording()
    if rec is not None:
        module, test = _current_module()
        rec.begin(test)
        key = _call_key(cmd, hint, flags, in_arrays, out_arrays, fmt, in_fmts, out_fmts)
        restored = rec.restore(list(in_arrays) + list(out_arrays))
    cache = {}

    def tensor_for(a, f):
        if a is None:
            return None
        if id(a) not in cache:
            cache[id(a)] = ref.RefTensor(a, f)
        return cache[id(a)]

    ins = [tensor_for(a, in_fmts[i] if in_fmts else fmt) for i, a in enumerate(in_arrays)]
    outs = [tensor_for(a, out_fmts[i] if out_fmts else fmt) for i, a in enumerate(out_arrays)]
    status = ref.cmd_exec(cmd, hint, flags, ins, outs)
    for t in cache.values():
        t.free()
    if rec is not None:
        rec.resample([a for a in restored if all(a is not o for o in out_arrays)])
        rec.record(module, key, status, out_arrays, whole)
    return status, out_arrays


def _known(got, want):
    """got and want as float64, without the positions a sampled stored reference output does not hold."""
    sg, sw = is_sampled(got), is_sampled(want)
    got64 = np.broadcast_to(np.asarray(got, dtype=np.float64), np.shape(want))
    want64 = np.asarray(want, dtype=np.float64)
    if not (sg or sw):
        return got64, want64
    m = np.ones(want64.shape, bool)
    if sw:
        m &= ~np.isnan(want64)
    if sg:
        m &= ~np.isnan(got64)
    return got64[m], want64[m]


def same(got, want):
    """np.array_equal, over the positions a sampled stored reference output holds."""
    if np.shape(got) != np.shape(want):
        return False
    g, w = _known(got, want)
    return w.size > 0 and np.array_equal(g, w)


def max_abs_diff(got, want):
    g, w = _known(got, want)
    return float(np.abs(g - w).max())


def max_abs(want):
    w = np.abs(np.asarray(want, dtype=np.float64))
    return float(np.nanmax(w) if is_sampled(want) else w.max())


def rel_err(got, want):
    """max |got - want| / max(|want|): the normalised error the fp32 tolerance of BASELINE.json (<= 1e-3) is applied to."""
    got, want = _known(got, want)
    denom = max(np.abs(want).max(), 1e-30)
    return float(np.abs(got - want).max() / denom)


def elem_rel_err(got, want, floor=1e-2):
    """Element-wise relative error max |got - want| / max(|want|, floor * max|want|): small outputs count with their own
    magnitude down to an absolute floor of `floor` x the largest reference value (below that, fp32 summation-order noise of
    the reference itself dominates)."""
    got, want = _known(got, want)
    scale = max(np.abs(want).max(), 1e-30)
    return float((np.abs(got - want) / np.maximum(np.abs(want), floor * scale)).max())


def assert_close(got, want, tol, what=""):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    held = got[~np.isnan(got)] if is_sampled(got) else got
    assert np.isfinite(held).all(), what + ": non-finite output"
    e = rel_err(got, want)
    assert e <= tol, "%s: normalised max error %.3e > %.1e" % (what, e, tol)


# ---- 16-bit tensors: bf16 travels as uint16 (numpy has no bfloat16), fp16 as numpy float16 ------------------------------
def to_bf16(a):
    """fp32 -> bf16 bits (uint16), round to nearest even."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    return r.reshape(np.shape(a))


def from_bf16(u):
    return (np.ascontiguousarray(u, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32).reshape(np.shape(u))


def round16(a, kind):
    """The fp32 values a 16-bit tensor of this kind (abi.CCV_16BF / abi.CCV_16F) actually holds."""
    return from_bf16(to_bf16(a)) if kind == abi.CCV_16BF else np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


def pack16(a, kind):
    return to_bf16(a) if kind == abi.CCV_16BF else np.asarray(a, np.float32).astype(np.float16)


def unpack16(u, kind):
    return from_bf16(u) if kind == abi.CCV_16BF else np.asarray(u, np.float16).astype(np.float32)


def gpu_exec16(nnc, cmd, hint, flags, in_arrays, out_arrays, kind, keep32=(), stream=None, in_fmts=None, out_fmts=None):
    """gpu_exec with fp32 numpy arrays travelling as 16-bit tensors of `kind`.  `keep32`: ids (id(array)) of operands that stay
    fp32 (batch-norm parameters / statistics, fp32 master weights of SGD).  Integer arrays travel unchanged.  The same array
    object in both lists is the same GPU tensor.  Returns (status, [fp32 output arrays])."""
    cache = {}

    def tensor_for(a, f=NHWC):
        if a is None:
            return None
        if id(a) not in cache:
            if a.dtype != np.float32 or id(a) in keep32:
                t = nnc.gpu_tensor(list(a.shape), f, NP_TO_CCV[a.dtype])
                t.upload(a)
            else:
                t = nnc.gpu_tensor(list(a.shape), f, kind)
                t.upload(pack16(a, kind))
            cache[id(a)] = t
        return cache[id(a)]

    ins = [tensor_for(a, in_fmts[i] if in_fmts else NHWC) for i, a in enumerate(in_arrays)]
    outs = [tensor_for(a, out_fmts[i] if out_fmts else NHWC) for i, a in enumerate(out_arrays)]
    status = nnc.cmd_exec(cmd, hint, flags, ins, outs, stream)
    if stream is not None:
        stream.wait()
    results = []
    for t in outs:
        if t is None:
            results.append(None)
        elif (t.params.datatype & 0xFF000) in (abi.CCV_16BF, abi.CCV_16F):
            results.append(unpack16(t.download(), t.params.datatype & 0xFF000))
        else:
            results.append(t.download())
    for t in cache.values():
        t.free()
    return status, results
