import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # build the native pieces once (no-ops when up to date; nvcc cross-compiles without a GPU)
    if shutil.which("nvcc"):
        import __graft_entry__
        __graft_entry__.load_builder().build_all()
    from oracle import build as obuild
    obuild.build_oracle_c()
    # METIS for the METIS tests: the package's own copy, else the one build() links into oracle/_ref
    import __graft_entry__
    if not os.path.exists(__graft_entry__.load_builder().METIS_LIB) and os.path.exists(obuild.ref_metis_path()):
        os.environ.setdefault("PGLB_LIBMETIS", obuild.ref_metis_path())


def pytest_collection_modifyitems(config, items):
    """`gpu`-marked tests need a CUDA device: skip them (instead of erroring) on a CPU box, so a plain
    `pytest tests/` is clean everywhere (ADVICE r1)."""
    try:
        import torch
        has_cuda = torch.cuda.is_available()
    except Exception:
        has_cuda = False
    if has_cuda:
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def kat():
    import json
    with open(os.path.join(GOLDEN, "kat.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def oracle_c():
    import ctypes
    from oracle import build as obuild
    return ctypes.CDLL(obuild.build_oracle_c())
