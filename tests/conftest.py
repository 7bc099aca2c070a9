"""pytest configuration: `gpu` marker, builds of the oracle and of the CUDA library, shared fixtures."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (runs on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle (test infrastructure; never used by the product path)."""
    from oracle import binding

    binding.build()
    return binding


_RECORDS = {}  # module -> test -> outputs of the compiled reference recorded in this session


@pytest.fixture
def reference(request):
    """The outputs of the reference's own sources (oracle/_ref) for this test, replayed from tests/golden/reference/;
    with SVO_RECORD_REFERENCE=DIR they are recorded from oracle/_ref into DIR instead (tests/reference_outputs.py)."""
    from tests import reference_outputs

    r = reference_outputs.Reference(request.node.module.__name__.rsplit(".", 1)[-1], request.node.name,
                                    os.environ.get("SVO_RECORD_REFERENCE") or None)
    yield r
    r.finish(_RECORDS)


def pytest_sessionfinish(session):
    if _RECORDS:
        from tests import reference_outputs

        reference_outputs.write(os.environ["SVO_RECORD_REFERENCE"], _RECORDS)


@pytest.fixture(scope="session")
def ctx():
    """A CUDA context of the product library; fails loudly when there is no GPU."""
    from rpg_svo_b200 import capi

    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def pair300():
    from rpg_svo_b200 import synth

    return synth.make_frame_pair(1000, n_feat=300, n_levels=5)
