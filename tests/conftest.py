import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _usable_cpus():
    """affinity capped by the cgroup CPU quota: the reference oracle (OpenMP) must not run 128 threads on a 16-CPU lease"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        a, b = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if a != "max":
            n = max(1, min(n, int(float(a) / float(b) + 0.5)))
    except Exception:
        pass
    return n


os.environ.setdefault("OMP_NUM_THREADS", str(_usable_cpus()))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture
def ref(request):
    """the compiled reference oracle's answers for this test, replayed from tests/golden/ref (oracle/tape.py);
    KB2_RECORD_REF=1 records them from oracle/_ref instead"""
    from oracle import tape
    test_id = f"{request.node.module.__name__}::{request.node.name}"
    session = tape.Recorder(test_id) if tape.recording() else tape.Player(test_id)
    yield tape.Ref(session)
    rep = getattr(request.node, "rep_call", None)
    if tape.recording() and rep is not None and rep.passed:
        session.save()


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_makereport(item, call):
    rep = (yield).get_result()
    setattr(item, "rep_" + rep.when, rep)


@pytest.fixture(scope="session")
def kb():
    import knowhere_b200
    return knowhere_b200
