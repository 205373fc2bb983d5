import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# GPU tests that exercise code changed after the last run on a B200 (DIO's ripple path, event rings, drop-in
# programs) run after the ones that were measured there: with `pytest -x` an early surprise must not hide the rest.
_RUN_LAST = ("golden_dio", "dio_path", "dio_decimated", "edge_cases", "long_48k", "legacy_api_and_analyze_host",
             "analyze_coded_host", "host_pipeline_chunking", "event_dense", "zero_tail_f0", "mirroring_ripple",
             "reference_examples", "cpp_batched")


def pytest_collection_modifyitems(config, items):
    items.sort(key=lambda it: 1 if ("gpu" in it.keywords and any(k in it.name for k in _RUN_LAST)) else 0)
    if _have_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture
def ref(request):
    """The unmodified reference's results for this test, replayed from tests/golden/reference; with WB_REF_RECORD
    set, the reference compiled into oracle/_ref runs and its results are stored (tests/refreplay.py)."""
    import refreplay
    record = os.environ.get("WB_REF_RECORD")
    if not record:
        return refreplay.Replayer(request.node)
    from refworld import RefWorld, REF_LIB
    if not os.path.exists(REF_LIB):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"])
    rec = refreplay.Recorder(RefWorld(REF_LIB), request.node,
                             refreplay.GOLDEN_DIR if record == "1" else os.path.abspath(record))
    request.addfinalizer(rec.save)
    return rec


@pytest.fixture
def ref_digests(request):
    """SHA-256 of the reference's results for the tests that compare bytes or bits with it (tests/refreplay.py);
    with WB_REF_RECORD set they are computed by the compiled reference (.live) and stored."""
    import refreplay
    record = os.environ.get("WB_REF_RECORD")
    if not record:
        return refreplay.Digests(request.node)
    from refworld import RefWorld, REF_LIB
    if not os.path.exists(REF_LIB):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"])
    d = refreplay.Digests(request.node, RefWorld(REF_LIB),
                          refreplay.GOLDEN_DIR if record == "1" else os.path.abspath(record))
    request.addfinalizer(d.save)
    return d


@pytest.fixture(scope="session")
def golden():
    import refreplay
    return refreplay.load_vaiueo2d()


@pytest.fixture(scope="session")
def emu():
    """Single-thread host emulation of the kernel sources (logic check without a GPU)."""
    from world_b200.api import World
    path = os.path.join(ROOT, "tests", "emu", "libworld_b200_emu.so")
    subprocess.check_call([os.path.join(ROOT, "tests", "emu", "build.sh")], stdout=subprocess.DEVNULL)
    # WB_EMU_LIB: an instrumented build of the same sources (e.g. -fsanitize=address, see tests/emu/README)
    return World(lib_path=os.environ.get("WB_EMU_LIB", path), array_module="numpy")


@pytest.fixture(scope="session")
def gpu_world():
    import torch
    from world_b200.api import World
    torch.cuda.set_device(0)
    return World(device=0)
