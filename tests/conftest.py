import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    """GPU tests are skipped (not failed) when no device is visible."""
    try:
        import torch
        have = torch.cuda.is_available()
    except Exception:
        have = False
    if have:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


PARITY_LOG = os.path.join(ROOT, "gpurun_out", "parity.jsonl")


def record_parity(case: str, **metrics):
    """Append the ACHIEVED error of a parity case to gpurun_out/parity.jsonl (copied to profiles/r02_parity.json after a
    GPU run): the judge reads achieved maxima, not just pass / fail."""
    import json
    try:
        os.makedirs(os.path.dirname(PARITY_LOG), exist_ok=True)
        with open(PARITY_LOG, "a") as f:
            f.write(json.dumps({"case": case, **{k: (float(v) if hasattr(v, "__float__") else v) for k, v in metrics.items()}}) + "\n")
    except OSError:
        pass
