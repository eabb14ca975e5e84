import os
import sys
import warnings

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def lookup_dir(tmp_path_factory):
    """Directory with the nine default lookup CSVs, byte-identical to the reference's."""
    from tests import lookups
    return lookups.write_default_lookups(str(tmp_path_factory.mktemp("lookups")))


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement oracle (built on demand)."""
    from oracle import oracle as O
    return O.Port()


@pytest.fixture(scope="session")
def ref():
    """The reference's own object code, if the prebuilt library is present."""
    from oracle import oracle as O
    if not O.Ref.available():
        pytest.skip("oracle/_ref/libgcn10_ref.so not present")
    return O.Ref()


@pytest.fixture(scope="session")
def reference(port):
    """What process_block() saves (``run_block``) and its window arithmetic (``window``): the reference's own object
    code where oracle/_ref is built, else the plain-C restatement, which the golden fixtures in tests/golden/ (outputs
    of that object code) pin to it.  The substitution is reported as a warning in the test summary."""
    from oracle import oracle as O
    if O.Ref.available():
        return O.Ref()
    warnings.warn("oracle/_ref/libgcn10_ref.so not present: expected rasters and windows come from the plain-C "
                  "restatement (oracle/cn_oracle.c), pinned to the reference by tests/golden/")
    return port


@pytest.fixture(scope="session")
def tables(port, lookup_dir):
    return port.load_tables(lookup_dir)


@pytest.fixture(scope="session")
def gpu_ctx(tables):
    """A libgcn10cuda context on cuda:0 with the default tables installed.  No fallback."""
    from gcn10_b200 import capi
    ctx = capi.Context(0)
    ctx.set_luts(tables)
    yield ctx
    ctx.close()
