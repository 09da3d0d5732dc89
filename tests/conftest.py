import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT, ROOT / "yolo-re_b200"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def gelan_c():
    """(nodes, nc, calibrated state_dict) of gelan-c from the oracle -- deterministic."""
    from oracle import gelan_ref as G
    nodes, nc = G.load_graph(ROOT / "configs/models/gelan-c.yaml")
    return nodes, nc, G.calibrated_state_dict(nodes, nc)


@pytest.fixture(scope="session")
def yolov9_c():
    from oracle import gelan_ref as G
    nodes, nc = G.load_graph(ROOT / "configs/models/yolov9-c.yaml")
    return nodes, nc, G.calibrated_state_dict(nodes, nc)


@pytest.fixture(scope="session", autouse=True)
def _oracle_built():
    """The oracle's C port is test infrastructure; build it on demand."""
    import subprocess
    so = ROOT / "oracle" / "_build" / "libnms_ref.so"
    if not so.exists():
        subprocess.check_call(["make", "-C", str(ROOT / "oracle")])
