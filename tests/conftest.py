import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")
    config.addinivalue_line("markers", "reference: runs the reference's own scripts from oracle/_ref/ (staged by build() where the reference tree is readable)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(skip_gpu)


@pytest.fixture(scope="session")
def checkpoints():
    from oracle import synth
    return synth.make_checkpoints(0)


@pytest.fixture(scope="session")
def gpu_models(checkpoints):
    """The three product modules, strict-loaded with the synthetic checkpoints, on cuda:0."""
    import torch
    from marconet_b200.models import networks
    dev = torch.device("cuda:0")
    out = {}
    for key, cls in (("tspgan", networks.TSPGAN), ("encoder", networks.TextContextEncoderV2), ("sr", networks.TSPSRNet)):
        m = cls()
        m.load_state_dict(checkpoints[key], strict=True)
        out[key] = m.eval().to(dev)
    return out
