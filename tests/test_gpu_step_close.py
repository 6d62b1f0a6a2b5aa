"""GPU: a step's counters are folded into `AsStats` once, whichever kernel gets there first.

A peer-connected handle (world 1) can fold in three places besides the finish kernel: the step kernel's last CTA (to
exchange the counters), `as_fold_stats`, and the exchange kernel behind a step left open.  A second fold would read
the emptied counter slots and overwrite the statistics with zeros.
"""
from __future__ import annotations

import ctypes as C

import pytest
import torch

from test_gpu_step_variants import QUIET_STEP, Replay, compare_stats, physics, to_views
from terms_oracle import STAT_FIELDS

pytestmark = pytest.mark.gpu

N = 1001


def launch_fused(mdp, views, actions, out, defer):
    """`as_step_fused` as `AllstepsMDP.step` issues it, without `finish_step`."""
    from allsteps_isaaclab_b200 import _cabi

    out.step_out.flags = _cabi.STEP_DEFER_FINISH if defer else 0
    _cabi.check(mdp.lib.as_step_fused(mdp.handle, C.byref(views.struct), actions.data_ptr(), actions.stride(0),
                                      C.byref(out.step_out), C.byref(out.reset_out), mdp._stream()), "as_step_fused")


@pytest.mark.parametrize("route", ["quiet-step-closed-by-fix-up", "deferred-step-closed-by-exchange"])
def test_fold_stats_after_a_fold_changes_nothing(route):
    """quiet-step-closed-by-fix-up: a step in which no env resets, launched to close itself -- its last CTA folds for
    the exchange and leaves the step to the fix-up.  deferred-step-closed-by-exchange: a step with resets launched with
    AS_STEP_DEFER_FINISH, closed by `finish_step()` without a global record, i.e. through the exchange kernel.  In both,
    `fold_stats()` before `finish_step()` must leave statistics, outputs and state as a twin handle that skips it."""
    from allsteps_isaaclab_b200.mdp import StepBuffers

    rp = Replay(N, seed=61)
    sc, orc = rp.sc, rp.orc
    twins = [rp.mdps[0], rp.new_handle()]  # twins[0] calls fold_stats()
    for mdp in twins:
        mdp.connect_self()
    outs = [StepBuffers(N, "cuda:0") for _ in twins]
    quiet = route.startswith("quiet")
    probe = QUIET_STEP if quiet else 0
    for step in range(probe + 1):
        phys = physics(sc, orc, step)
        m, n = sc.reset_uniforms(step)
        orc.step(phys, phys["actions"], m, n, None)
        for i, (mdp, out) in enumerate(zip(twins, outs)):
            views, keep = to_views(phys, rp.origins, sc.body_indices)
            if step < probe:
                mdp.step(views, keep["actions"], out)
                continue
            launch_fused(mdp, views, keep["actions"], out, defer=not quiet)
            if i == 0:
                mdp.fold_stats()
            mdp.finish_step()
        torch.cuda.synchronize()
    assert (orc.stats["n_reset"] == 0) == quiet, f"{route}: {orc.stats['n_reset']} resets"
    folded, plain = (m.read_stats() for m in twins)
    assert plain["sum_target_index"] > 0 and plain["n_advanced"] > 0, plain
    bad = {k: (folded[k], plain[k]) for k in STAT_FIELDS if folded[k] != plain[k]}
    assert not bad, f"{route}: AsStats (fold_stats, plain) differ: {bad}"
    for mdp in twins:
        compare_stats(mdp.read_stats(), orc, route)
    for name in ("obs", "reward", "terminated", "time_out", "n_reset"):
        assert torch.equal(getattr(outs[0], name), getattr(outs[1], name)), f"{route}: {name}"
    a, b = (m.export_state() for m in twins)
    for k in a:
        assert torch.equal(a[k], b[k]), f"{route}: state {k}"
