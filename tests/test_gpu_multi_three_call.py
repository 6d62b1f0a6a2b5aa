"""World-size-2 checks of the global 3-call mode (tools/three_call_peer_check.py): every shard of a sharded 3-call run
equals its slice of one handle holding all envs.  With two GPUs visible the ranks run one per GPU over NCCL; on a
one-GPU box they run as two processes sharing the GPU (CUDA IPC peer memory works between processes on one device;
the tool's gathers then go through gloo), so the check is never skipped."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(port, env_extra, timeout=900):
    env = dict(os.environ, THREE_CALL_CHECK_BACKEND="nccl" if torch.cuda.device_count() >= 2 else "gloo", **env_extra)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "tools", "three_call_peer_check.py")]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)


@pytest.mark.gpu
def test_sharded_three_call_run_equals_one_handle():
    """Outputs, state, levels, bins, stones and statistics of every shard equal the single handle's at every step,
    histograms right after every pass 1 -- through steps where only one rank resets, steps where nobody does, a
    promotion, a reset outside a step, both id routes, and `StandaloneAllstepsEnv(..., distributed=True)`."""
    res = _run(29551, {})
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "three_call_peer_check OK" in res.stdout


@pytest.mark.gpu
def test_shard_local_three_call_parts_from_one_handle_where_one_rank_resets():
    """Without the mode (the shards run shard-local) the same scenario parts from the single handle first at a step
    in which only one rank has resets: the other rank takes pass 2 back although the reference runs it for every env
    (DRL:359-360).  This is what the test above covers."""
    res = _run(29553, {"THREE_CALL_CHECK_MODE": "local"})
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    m = re.search(r"LOCAL DIFFERS first at step (\d+) .*?, (\w+ \w+) reset: (.*)", res.stdout)
    assert m and "outside a step" not in res.stdout, res.stdout[-3000:]
    assert m.group(2) == "one rank", m.group(0)
    assert "obs" in m.group(3).split(", "), m.group(0)
