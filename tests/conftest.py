import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
WEIGHTS = os.path.join(ROOT, "weights")
# optional checkout of the reference project (MerlinPCarson/WakeWord-Detection): the tests that compare with its
# own files run only when it is given; everything else compares with the vectors under tests/golden/
REFERENCE = os.environ.get("WWB_REFERENCE", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_weights(name):
    from wakeword_detection_b200 import weights as W
    typ = "Wavenet" if name.lower().startswith("wavenet") else "CRNN"
    return W.load_model_dir(os.path.join(WEIGHTS, name), typ)


@pytest.fixture(scope="session")
def w_crnn():
    return load_weights("CRNN")


@pytest.fixture(scope="session")
def w_crnn_softmax():
    return load_weights("CRNN_arik_original")


@pytest.fixture(scope="session")
def w_wavenet():
    return load_weights("Wavenet")


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(GOLDEN, "reference_glue.npz"))


@pytest.fixture(scope="session")
def wake_mel():
    return {k: np.load(os.path.join(GOLDEN, "wake_%s_mel.npy" % k)) for k in ("crnn", "wavenet")}


@pytest.fixture(scope="session")
def wake_pcm():
    return {k: np.load(os.path.join(GOLDEN, "wake_%s_pcm.npy" % k)) for k in ("crnn", "wavenet")}


_ENGINES = {}


def get_engine(name, precision="tc"):
    from wakeword_detection_b200 import _cabi
    key = (name, precision)
    if key not in _ENGINES:
        _ENGINES[key] = _cabi.Engine(load_weights(name), 0, precision)
    return _ENGINES[key]
