import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.hookimpl(tryfirst=True)
def pytest_cmdline_main(config):
    """The CPU suite (`-m "not gpu"`: ~110 tests, most of them world-2/4 gloo runs that spend their
    time in process start-up) runs on 4 pytest-xdist workers when xdist is installed: 3.5 instead of
    8 minutes on 8 cores.  Every multi-rank test rendezvouses on its own free port (tests/_procs.py),
    so workers cannot collide.  GPU runs (`-m gpu`) stay serial — one GPU, timing-sensitive — and so
    does anything with an explicit `-n`, a `-k` selection or EDB_TEST_WORKERS=0."""
    opt = config.option
    if os.environ.get("PYTEST_XDIST_WORKER") or hasattr(config, "workerinput"):
        return None
    if getattr(opt, "markexpr", "").strip() != "not gpu" or getattr(opt, "keyword", ""):
        return None
    if not hasattr(opt, "numprocesses") or opt.numprocesses is not None:
        return None   # xdist missing / disabled, or the caller chose
    if getattr(opt, "collectonly", False) or getattr(opt, "usepdb", False):
        return None
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    workers = min(int(os.environ.get("EDB_TEST_WORKERS", "4")), cores // 2)
    if workers >= 2:
        opt.numprocesses = workers   # xdist's own cmdline hook (runs after this one) does the rest
    return None


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 GPUs on the box")
    config.addinivalue_line("markers", "refonly: needs the reference source tree (EASYDIST_REFERENCE)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
