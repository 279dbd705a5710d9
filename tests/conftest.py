import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
# every frequency-masking iteration also runs the device histogram pass and checks the
# host-maintained symbol histograms against it (search.cc, encoded_size)
os.environ.setdefault("GB200_CHECK_HOST_HIST", "1")
# The CPU port runs its emulated kernels as OpenMP loops, thousands of tiny parallel regions per
# image: with spinning waits they crawl whenever the box is busy (another job on one core is
# enough), so the workers sleep instead and the team stays small.
os.environ.setdefault("OMP_WAIT_POLICY", "passive")
os.environ.setdefault("OMP_NUM_THREADS", str(max(1, min(4, len(os.sched_getaffinity(0))))))
# GB200_RECORD_REFERENCE=1: the tests that ask the reference get the live build in oracle/_ref and
# its answers are written to tests/golden/reference_answers.json (tests/refanswers.py); only those
# tests run, the GPU ones on the CPU port, which computes the product's bits.  Two GPU tests fail
# there, harmlessly: test_cuda_cli runs the CUDA command-line tool (test_port_cli asks the same
# questions) and test_process_matches_reference_256 counts kernel launches after its questions.
RECORD = os.environ.get("GB200_RECORD_REFERENCE") == "1"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def pytest_collection_modifyitems(config, items):
    if RECORD:
        keep = [it for it in items if "ref" in getattr(it, "fixturenames", ())]
        config.hook.pytest_deselected(items=[it for it in items if it not in keep])
        items[:] = keep


@pytest.fixture(scope="session")
def port_lib():
    """CPU restatement of the hot path (oracle/_build/libguetzli_port.so)."""
    import guetzli_b200 as gb
    path = os.path.join(ROOT, "oracle", "_build", "libguetzli_port.so")
    if not os.path.exists(path):
        import __graft_entry__
        __graft_entry__.build()
    return gb.load_library(path)


@pytest.fixture(scope="session")
def cuda_lib(request):
    """The product library; requires a GPU."""
    if RECORD:
        return request.getfixturevalue("port_lib")
    import guetzli_b200 as gb
    lib = gb.load_library()
    assert lib.gb200_backend_name() == b"cuda-sm_100a"
    assert lib.gb200_device_count() >= 1, "no CUDA device visible"
    return lib


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference: its recorded answers (tests/refanswers.py), or while recording
    the live build in oracle/_ref."""
    import refanswers
    if not RECORD:
        yield refanswers.Replay()
        return
    import reflib
    if not reflib.available():
        pytest.exit("GB200_RECORD_REFERENCE=1 needs the reference built into oracle/_ref", returncode=2)
    rec = refanswers.Recorder()
    yield rec
    rec.save()
