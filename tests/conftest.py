import base64
import gzip
import json
import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

GOLDEN = os.path.join(REPO, "tests", "golden")


def pytest_collection_modifyitems(config, items):
    """gpu-marked tests are skipped (not failed) on a machine without a CUDA device."""
    try:
        import torch
        have = torch.cuda.is_available()
    except Exception:  # noqa: BLE001
        have = False
    asked = config.getoption("-m") or ""
    if have or ("gpu" in asked and "not gpu" not in asked):
        return                    # with `-m gpu` on a box without a device the tests FAIL loudly, as they should
    skip = pytest.mark.skip(reason="no CUDA device (run with -m gpu on a B200)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")


def load_golden(name):
    with open(os.path.join(GOLDEN, name)) as fh:
        return json.load(fh)


def file_bytes(spec):
    """Decode one file entry of a golden case."""
    if "text" in spec:
        return spec["text"].encode("utf-8")
    if "gzb64" in spec:
        return gzip.decompress(base64.b64decode(spec["gzb64"]))
    return base64.b64decode(spec["b64"])


def materialize(files, directory):
    for name, spec in files.items():
        with open(os.path.join(str(directory), name), "wb") as fh:
            fh.write(file_bytes(spec))


@pytest.fixture
def in_tmp(tmp_path):
    """chdir into a scratch directory for the duration of a test."""
    old = os.getcwd()
    os.chdir(str(tmp_path))
    try:
        yield tmp_path
    finally:
        os.chdir(old)


NO_REFERENCE = "the original tagdigger is not staged in oracle/_ref (oracle/stage_ref.py)"


def have_reference():
    from oracle import stage_ref
    return stage_ref.staged()


def import_reference():
    """The live reference: the unmodified copy staged in oracle/_ref."""
    from oracle import stage_ref
    return stage_ref.import_ref()
