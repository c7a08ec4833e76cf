import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # checker libraries: the port always builds; the reference only where its source tree is present (oracle/Makefile REF)
    try:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"], check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    except Exception:
        pass


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture
def ref(request):
    """The unmodified reference: the library itself where oracle/_ref/libdsv1ref.so is built, otherwise its recorded
    results (tests/refdigest.py) checked against the library the test exercises."""
    import dsvlibs
    import refdigest
    if dsvlibs.have_ref():
        lib = dsvlibs.ref()
        return refdigest.Recorder(lib) if os.environ.get("DSV1_RECORD_REFERENCE") == "1" else lib
    for name in ("gpu", "emu", "port"):
        if name in request.fixturenames:
            return refdigest.RecordedReference(request.getfixturevalue(name))
    raise LookupError("the ref fixture needs the gpu, emu or port fixture beside it")


@pytest.fixture(scope="session")
def port():
    import dsvlibs
    return dsvlibs.port()


@pytest.fixture(scope="session")
def gpu():
    import dsvlibs
    return dsvlibs.gpu()
