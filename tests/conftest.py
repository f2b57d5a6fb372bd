import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    try:  # fp32 torch references on the GPU must not silently run in TF32
        import torch
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
    except Exception:
        pass
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import io
    import lzma
    import torch
    sys.path.insert(0, GOLDEN)
    import golden_inputs

    def load(name):
        path = os.path.join(GOLDEN, name)
        if os.path.exists(path + ".xz"):      # a fixture whose outputs alone pass 1 MB is stored xz-compressed
            with lzma.open(path + ".xz") as f:
                path = io.BytesIO(f.read())
        fixture = torch.load(path, map_location="cpu", weights_only=False)
        return golden_inputs.attach(name, fixture)   # inputs drawn from their seeds again, checked against a digest
    return load
