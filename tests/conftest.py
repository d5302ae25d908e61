import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement oracle (always buildable: gcc only)."""
    import oracle
    if not os.path.exists(oracle.PORT_SO):
        oracle.build(port=True, ref=False)
    return oracle.Port()


@pytest.fixture(scope="session")
def reference_outputs():
    """What the compiled reference returned on the tests' random inputs
    (recorded by tests/golden/make_reference_outputs.py)."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_outputs.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def checker(port):
    """Strongest checker available: compiled reference if present, else the port."""
    import oracle
    if oracle.Ref.available():
        try:
            return oracle.Ref()
        except OSError:
            pass
    return port


@pytest.fixture(scope="session")
def hb():
    lib = os.path.join(ROOT, "hexl_b200", "lib", "libhexl_b200.so")
    if not os.path.exists(lib):
        # the package refuses to import without its library; run its build script directly
        import importlib.util
        spec = importlib.util.spec_from_file_location("_hexl_b200_build", os.path.join(ROOT, "hexl_b200", "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    import hexl_b200
    return hexl_b200


@pytest.fixture(scope="session")
def kats():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_kats.json")) as f:
        return json.load(f)
