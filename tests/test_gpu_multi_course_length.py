"""World-size-2 check of the global 3-call mode at courses of 12 stones (tools/three_call_peer_check.py --num-steps 12):
every shard equals its slice of one handle holding all envs, as tests/test_gpu_multi_three_call.py checks at 20 (two
GPUs over NCCL, or two processes sharing one GPU over gloo)."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_sharded_three_call_run_equals_one_handle_at_12_stones():
    env = dict(os.environ, THREE_CALL_CHECK_BACKEND="nccl" if torch.cuda.device_count() >= 2 else "gloo")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29557",
           os.path.join(ROOT, "tools", "three_call_peer_check.py"), "--num-steps", "12"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "three_call_peer_check OK" in res.stdout and "12 stones" in res.stdout
