import importlib.util
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_pkg():
    """import the package whose directory name contains a dot"""
    if "welle_io_b200" in sys.modules:
        return sys.modules["welle_io_b200"]
    d = os.path.join(ROOT, "welle.io_b200")
    spec = importlib.util.spec_from_file_location("welle_io_b200", os.path.join(d, "__init__.py"), submodule_search_locations=[d])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["welle_io_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="session")
def pkg():
    return load_pkg()


@pytest.fixture(scope="session")
def oracle():
    from oracle.bind import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    """the reference build (oracle/_ref) where it can be built, else its results recorded in tests/golden/ref_calls.npz;
    DABB_RECORD_REF=<file> records the live reference's results of this session into <file>"""
    import refcalls
    from oracle.bind import Ref, build_ref
    if not Ref.available():
        build_ref()
    if not Ref.available():
        yield refcalls.ReplayRef()
        return
    path = os.environ.get("DABB_RECORD_REF")
    if not path:
        yield Ref()
        return
    rec = refcalls.RecordingRef(Ref())
    yield rec
    rec.save(path)
