"""GPU (two devices): the C-level multi-GPU entry, dctz_gpu_compress_slab_comm -- statistics exchange and QT table
reduction over NCCL inside the library, driven by a plain C program with one host thread per rank
(tests/c/slab_comm_test.c -> dctz_b200/bin/slab-comm-test).  Skipped on a single-GPU box."""
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_ranks_over_nccl_from_c():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    exe = os.path.join(ROOT, "dctz_b200", "bin", "slab-comm-test")
    assert os.path.exists(exe), "run __graft_entry__.build()"
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and "slab_comm_test OK" in p.stdout, p.stdout[-2000:] + p.stderr[-2000:]
    assert "mode EC: 2 ranks over NCCL == one GPU" in p.stdout and "mode QT: 2 ranks over NCCL == one GPU" in p.stdout
