import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch

    has_gpu = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture
def mjcf_file(tmp_path):
    def _write(xml: str, name: str = "model.xml") -> str:
        p = tmp_path / name
        p.write_text(xml)
        return str(p)

    return _write


def pytest_sessionfinish(session, exitstatus):
    """B200_PARITY_STATS=<path>: dump the measured error distributions of the parity tests (tests/parity_util.check_envelope)."""
    path = os.environ.get("B200_PARITY_STATS")
    if path:
        import json

        from tests.parity_util import PARITY_STATS

        if PARITY_STATS:
            os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
            json.dump(PARITY_STATS, open(path, "w"), indent=1, sort_keys=True)
