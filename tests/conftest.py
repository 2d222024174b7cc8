import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def locked_make(directory, *targets, env=None, jobs=None):
    """`make` under an exclusive file lock: pytest-xdist workers would otherwise rebuild the same library at the same time
    (one of them then loads a half-written .so)."""
    import fcntl, subprocess
    os.makedirs(directory, exist_ok=True)
    with open(os.path.join(directory, ".build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        try:
            cmd = ["make", "-C", directory, "-s"] + (["-j", str(jobs)] if jobs else []) + list(targets)
            subprocess.check_call(cmd, env={**os.environ, **(env or {})})
        finally:
            fcntl.flock(lk, fcntl.LOCK_UN)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    import oracle as o
    o.build()
    return o
