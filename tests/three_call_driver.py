"""Test infrastructure: one env step through the 3-call path (`pass1` -> `reset` -> `pass2`, or `no_reset`), with the
test playing PhysX between the calls, and the exact comparison of two handles' results after it.  Shared by
tests/test_gpu_three_call_peers.py and tools/three_call_peer_check.py."""
from __future__ import annotations

import torch

from test_gpu_three_call_curriculum import _physx_writes

OUTPUTS = ("obs", "reward", "terminated", "time_out", "dones", "final_obs")


def three_call_step(mdp, views, keep, out, origins, ep_len, device_list, after_pass1=None):
    """DRL:351-375 on `mdp`: `ep_len` (the DirectRLEnv counter) is advanced in place; `keep` (the tensors behind
    `views`) receives the PhysX writes of `_reset_idx`.  device_list: `reset(None)` takes the ids pass 1 compacted on
    the device, and the following `pass2` closes the step whether or not the list is empty; otherwise the ids come
    from `dones` on the host and an empty list means `no_reset()`.  Returns (reset ids in ascending order, the
    permutation that sorts the reset rows of `out` into that order)."""
    ep_len += 1  # DRL:351
    mdp.pass1(views, keep["actions"], out, episode_length=ep_len)
    if after_pass1 is not None:
        after_pass1()
    if device_list:
        mdp.reset(origins, None, out, episode_length=ep_len)
        n = int(out.n_reset.item())  # (the test plays PhysX: it needs the ids on the host side)
        ids = out.reset_ids[:n].long()
        _physx_writes(keep, ids, out, n)
        mdp.pass2(views, out)
        order = ids.argsort()
        return ids[order], order
    ids = out.dones.nonzero().squeeze(-1)  # DRL:359
    if len(ids):
        mdp.reset(origins, ids, out, episode_length=ep_len)
        _physx_writes(keep, ids, out, len(ids))
        mdp.pass2(views, out)
    else:
        mdp.no_reset()  # DRL:360
    return ids, torch.arange(len(ids), device=ids.device)


def reset_rows(out, order):
    """The start-pose rows of a step's reset envs in ascending env order: (k, 13 + 21 + 21)."""
    k = len(order)
    return torch.cat((out.reset_root_state[:k], out.reset_joint_pos[:k], out.reset_joint_vel[:k]), -1)[order]


def assert_same_step(a, b, what, rows_a=None, rows_b=None):
    """Bit-equality of two handles' step outputs (`StepBuffers`), state in the reference layout (levels and stones
    included), grid bins and, if given, reset rows.  `a` / `b`: (mdp, out)."""
    (ma, oa), (mb, ob) = a, b
    for name in OUTPUTS:
        x, y = getattr(oa, name), getattr(ob, name)
        if x is not None:
            assert torch.equal(x, y), f"{what}: {name} differs"
    if rows_a is not None:
        assert torch.equal(rows_a, rows_b), f"{what}: reset rows differ"
    sa, sb = ma.export_state(), mb.export_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), f"{what}: state {k} differs"
    if ma.grid_bins:
        assert torch.equal(ma.grid_state()[0], mb.grid_state()[0]), f"{what}: grid bins differ"
