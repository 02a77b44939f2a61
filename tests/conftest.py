import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run by the driver with -m gpu)")
    # tests/test_emulated_gpu_suite.py re-runs the gpu-marked parity tests on the CPU box in a child pytest whose
    # package is pointed at the emulated build of the library (tests/simt/library_emul.cc). Test infrastructure only:
    # the variable is read here, never by the package.
    emulated = os.environ.get("AMB_TEST_EMULATED_LIB")
    if emulated:
        from gr_air_modes_b200 import _lib
        _lib.LIB_PATH, _lib._lib = emulated, None


@pytest.fixture(scope="session")
def port():
    from oracle import cpu_oracle
    return cpu_oracle.Port()


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference objects, replayed from tests/golden/ref_results.json.xz. With AMB_TEST_RECORD_REF=1
    (tests/golden/make_ref_golden.py) the live objects answer instead and the session's calls are recorded."""
    from helpers import RecordedRef
    if os.environ.get("AMB_TEST_RECORD_REF") == "1":
        from oracle import cpu_oracle
        rec = RecordedRef(cpu_oracle.Ref())
        yield rec
        rec.save()
    else:
        yield RecordedRef()
