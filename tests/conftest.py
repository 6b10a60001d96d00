"""pytest configuration: `gpu` marker, import paths, shared fixtures.

CPU suite  : python -m pytest tests -x -q -m "not gpu"   (oracle vs golden, host logic, C-ABI symbols)
GPU suite  : python -m pytest tests -x -q -m gpu          (parity of the CUDA path, through the C ABI)
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def _ensure_built():
    import blinky_b200 as bb
    from oracle import pyoracle

    if not (os.path.exists(bb.LIB_PATH) and pyoracle.Restatement.available()):
        import __graft_entry__

        __graft_entry__.build()


@pytest.fixture(scope="session")
def bb():
    _ensure_built()
    import blinky_b200

    blinky_b200.load_library()
    return blinky_b200


@pytest.fixture(scope="session")
def palette(bb):
    return bb.synthetic_palette()


@pytest.fixture(scope="session")
def restate(bb):
    from oracle.pyoracle import Restatement

    assert Restatement.available(), "oracle/liboracle.so missing: run __graft_entry__.build()"
    return Restatement()


@pytest.fixture(scope="session")
def script_dir(bb):
    """directory whose lua-scripts/ both the product and the compiled reference read in tests:
    the repo's own script set (the reference's scripts are only used by the tests that say so)"""
    return bb.SCRIPT_DIR


def _gpu_run(config) -> bool:
    """True when this is the GPU suite (`-m gpu`): there a missing checker is a failure, not a skip"""
    expr = (config.getoption("markexpr", "") or "").replace(" ", "")
    return "gpu" in expr and "notgpu" not in expr


@pytest.fixture(scope="session")
def ref(bb, palette, script_dir):
    """the compiled UNMODIFIED reference (oracle/_ref), built only where the reference checkout is at
    hand.  Comparisons with it run against tests/golden/reference_live.json; only the tests that check
    the reference binary itself need it."""
    from oracle.pyoracle import RefOracle

    if not RefOracle.available():
        pytest.skip("oracle/_ref/libblinky_ref.so not built (needs the reference checkout at build time)")
    return RefOracle.get(script_dir, palette)


@pytest.fixture()
def host(bb, palette):
    """host-only product context (no GPU)"""
    fe = bb.Fisheye(device=None, palette=palette)
    yield fe
    fe.close()


@pytest.fixture(scope="session")
def cuda_device(request):
    import torch

    if not torch.cuda.is_available():
        if _gpu_run(request.config):
            pytest.fail("-m gpu was asked for but torch sees no CUDA device")
        pytest.skip("no CUDA device")
    return 0


def pytest_collection_modifyitems(config, items):
    # gpu tests must not silently pass on a box without a GPU
    pass


ALL_LENSES = ["cube", "cubestereo", "cylinder", "debug", "eckert1", "eckert4", "eckert5", "equirect", "fahey",
              "fisheye1", "fisheye2", "gallstereo", "gins8", "gumby", "hammer", "kavrayskiy7", "larrivee", "mercator",
              "miller", "mollweide", "panini", "polyconic", "quincuncial", "rectilinear", "sinusoidal",
              "stereographic", "vandergrinten", "wagner6", "winkel1", "winkel2", "winkeltripel"]
ALL_GLOBES = ["cube", "cube_corner", "cube_edge", "fast", "tetra", "trism"]


def sha(a: np.ndarray) -> str:
    import hashlib

    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
