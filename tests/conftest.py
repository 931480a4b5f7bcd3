import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "ref: needs oracle/_ref/libccv_ref.so (the compiled reference)")


def _has_gpu():
    try:
        from ccv_b200 import nnc
        return nnc.lib().ccv_nnc_device_count(nnc.CCV_STREAM_CONTEXT_GPU) > 0
    except Exception:
        return False


@pytest.fixture(scope="session")
def gpu():
    """The GPU tests must run the native library: fail (not skip) if it cannot be loaded on a GPU box."""
    from ccv_b200 import nnc
    nnc.init()
    if not _has_gpu():
        pytest.skip("no CUDA device")
    return nnc


def _usable_cpus():
    """CPUs this process may actually use: the affinity mask, cut by a cgroup CPU quota when there is one (a container on a 128-thread
    host is often allowed far fewer; OpenMP would still start 128 spinning threads per parallel region)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]  # cgroup v2
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())  # cgroup v1
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return max(1, n)


@pytest.fixture(scope="session")
def ref():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import ref as r
    if not r.available():
        # the outputs the compiled reference produced for these tests, stored under tests/golden/cpu_ref (tests/util.py)
        from tests.util import StoredRef
        return StoredRef()
    r.ref()
    # the parity cases are small: a handful of OpenMP threads serves them better than one per hardware thread of a large host (the GPU
    # suite spent most of its time in oversubscribed CPU_REF parallel regions); results do not depend on the count
    r.set_num_threads(min(16, _usable_cpus()))
    return r
