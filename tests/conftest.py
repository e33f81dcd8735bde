import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def ref_configs(tmp_path_factory):
    """The reference's config YAMLs (tests/golden/ref_configs.json) written out in their original layout, so that _BASE_ and
    MASKDINO.CONFIG_PATH resolve as they do in the reference tree.  Returns the configs directory."""
    import json
    import yaml
    with open(os.path.join(GOLDEN, "ref_configs.json")) as f:
        g = json.load(f)
    root = tmp_path_factory.mktemp("reference")
    for rel, d in g["files"].items():
        p = root / rel
        p.parent.mkdir(parents=True, exist_ok=True)
        p.write_text(yaml.safe_dump(d))
    return root / g["root"]


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")
