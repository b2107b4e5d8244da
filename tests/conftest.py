import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "reference: needs /root/reference (build container only)")


REFERENCE = "/root/reference"
needs_reference = pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="/root/reference not present")


@pytest.fixture(scope="session")
def reference_assets(tmp_path_factory):
    """The reference's robot descriptions (tests/golden/reference_assets.tar.xz) unpacked: an asset root laid out as its assets/."""
    import tarfile
    root = tmp_path_factory.mktemp("reference_assets")
    with tarfile.open(os.path.join(GOLDEN, "reference_assets.tar.xz")) as tar:
        tar.extractall(root, filter="data")
    return str(root)


@pytest.fixture(scope="session")
def reference_cfg():
    """The reference's task configs and PPO hyper-parameters (tests/golden/reference_cfg.json)."""
    import json
    with open(os.path.join(GOLDEN, "reference_cfg.json")) as f:
        return json.load(f)
