"""World-size-2 check of the grid curriculum's global histograms near the top of their uint32 counters: every shard
starts a few counts below 2^32 - 1, the summed outcomes of each step halve bins (the fold), and every shard must still
equal one handle holding all envs -- bins, stones, histograms.  Run like tests/test_gpu_multi.py: one rank per GPU over
NCCL with two GPUs, two processes sharing the GPU (CUDA IPC peer memory, all-reduce through gloo) with one."""
import pytest
import torch

from test_gpu_multi import _run


@pytest.mark.gpu
def test_global_histograms_fold_identically_on_every_shard():
    backend = "nccl" if torch.cuda.device_count() >= 2 else "gloo"
    res = _run(29547, {"PEER_CHECK_BACKEND": backend, "PEER_CHECK_GRID": "7", "PEER_CHECK_ENVS": "3000",
                       "PEER_CHECK_STEPS": "8", "PEER_CHECK_NEAR_TOP": "1"})
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "peer_check OK" in res.stdout and "grid 7x7 near the top of the counters" in res.stdout
