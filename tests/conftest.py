import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# a checkout of the upstream soft-grip repository (its data/gripper MJCF files); the tests that read it skip without it
REFERENCE = os.environ.get("SOFTGRIP_REFERENCE", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def pkg(sub=None):
    return importlib.import_module("soft-grip_b200" + ("." + sub if sub else ""))


@pytest.fixture(scope="session")
def mjcf():
    return pkg("mjcf")


@pytest.fixture(scope="session")
def batched():
    return pkg("batched")


@pytest.fixture(scope="session")
def oracle():
    from oracle import sgoracle
    sgoracle.build()
    return sgoracle


def blob_path(name):
    return os.path.join(GOLDEN, name + ".sgm")


@pytest.fixture(scope="session")
def make_world(oracle, mjcf, batched):
    cache = {}

    def _make(name, k=700.0):
        if name not in cache:
            blob = open(blob_path(name), "rb").read()
            cache[name] = (oracle.OracleModel(blob), mjcf.load_blob(blob))
        om, model = cache[name]
        w = oracle.OracleWorld(om)
        w.set_geom_mask(batched.geom_name_mask(model.names["geom"], "OBJ", ("g12", "g2")))
        if k is not None:
            w.set_stiffness(k)
        return w
    return _make


@pytest.fixture(scope="session")
def torch_cuda():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch
