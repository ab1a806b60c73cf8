import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on a B200 via gpurun)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def ref_model_dir(tmp_path_factory):
    """The reference's 2M-parameter test checkpoint (tests/models/llama-2m-fresh there), rebuilt from
    tests/golden/llama-2m-fresh.  Its config files and safetensors header are stored verbatim; the 1 MB of fresh-init
    weights are redrawn the way HF initialises them (norm weights 1, matrices N(0, 0.02)) from a fixed numpy seed."""
    import json
    import shutil
    import struct

    import numpy as np

    src = os.path.join(ROOT, "tests", "golden", "llama-2m-fresh")
    dst = tmp_path_factory.mktemp("llama-2m-fresh")
    for name in ("config.json", "generation_config.json"):
        shutil.copy(os.path.join(src, name), dst / name)
    with open(os.path.join(src, "model.safetensors.header.json"), "rb") as f:
        header = f.read()
    tensors = sorted((v["data_offsets"], v["shape"]) for k, v in json.loads(header).items() if k != "__metadata__")
    rng = np.random.default_rng(0)
    data = bytearray()
    for (begin, end), shape in tensors:
        assert begin == len(data) and end - begin == 4 * int(np.prod(shape))
        w = np.ones(shape, np.float32) if len(shape) == 1 else rng.normal(0.0, 0.02, shape).astype(np.float32)
        data += w.astype("<f4").tobytes()
    (dst / "model.safetensors").write_bytes(struct.pack("<Q", len(header)) + header + bytes(data))
    return str(dst)
