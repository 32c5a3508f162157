"""Split files identical across GPU counts (needs >= 2 CUDA devices; skipped on a one-GPU box).

Runs scripts/multigpu_split_check.py at world = every visible GPU: barcode_splitter_script under torchrun
splits one library file (plain LF, CRLF, BGZF) on every rank at once, and every output file's md5 and
rank 0's output must equal the single-process run's."""

import os
import subprocess
import sys

import pytest

from test_multigpu import REPO, _device_count

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(_device_count() < 2, reason="needs at least two GPUs")
def test_split_files_identical_across_gpu_counts():
    n = min(_device_count(), 8)
    p = subprocess.run([sys.executable, os.path.join(REPO, "scripts", "multigpu_split_check.py"), str(n)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, universal_newlines=True, timeout=1500)
    assert p.returncode == 0, p.stdout[-4000:]
    assert "MISMATCH" not in p.stdout and p.stdout.count(" OK") == 3, p.stdout[-4000:]
