"""Data-parallel parity on real GPUs (skipped on a 1-GPU box): 2 ranks over NCCL vs the
single-process oracle on the full batch."""
import pytest

from support import gpu_count, run_two_ranks

pytestmark = pytest.mark.gpu


def test_two_rank_training_equals_full_batch_oracle():
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = run_two_ranks("dist_worker.py", timeout=150)
    assert "DIST_OK world=2" in out
    assert "GRAPH_DIST_OK world=2" in out
    assert "CHUNKED_DIST_OK world=2" in out
