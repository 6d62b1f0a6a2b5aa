"""Device time of one env step on the 3-call path -- as_step_pass1 -> as_reset(device-side list) -> as_step_pass2, the
calls the DirectRLEnv hooks and the manager terms make around PhysX -- with the pitch x yaw grid curriculum off and on
(11 x 11 bins), on the chained synthetic workload (development tool, not the bench).

    python tools/three_call_grid_probe.py [N ...] [--steps K] [--repeats R]

Prints the card's name and power limit first: a time belongs to the card it was measured on.  Each configuration is
timed R times, off and on alternating, with CUDA events around K steps (the cycle's state rewind every 8 steps,
stone rows included, is the same in both), after a warm-up over two whole cycles.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from allsteps_isaaclab_b200 import synthetic as syn  # noqa: E402
from allsteps_isaaclab_b200.config import AllstepsCfg  # noqa: E402
from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers  # noqa: E402
from allsteps_isaaclab_b200.workload import ChainedWorkload  # noqa: E402

PERIOD = 8


def card() -> str:
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return f"{name} ({q[0]})" if q else name
    except (OSError, subprocess.TimeoutExpired):
        return f"{name} (power limit not readable)"


def make(N: int, grid_bins: int):
    cfg = AllstepsCfg()
    dev = torch.device("cuda:0")
    origins = syn.env_origins_grid(N, cfg.env_spacing).to(dev)
    mdp = AllstepsMDP(N, device=dev, seed=1, grid_bins=grid_bins)
    mdp.generate_stones(origins)
    st0 = syn.random_mdp_state(cfg, N, torch.Generator().manual_seed(1))
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                          "episode_length_buf", "potentials")})
    out = StepBuffers(N, dev)
    ep_len = torch.zeros(N, dtype=torch.int64, device=dev)
    calls = [0]

    def three_call(m, v, d, o):
        if calls[0] % PERIOD == 0:  # the cycle starts again: so does DirectRLEnv's episode counter
            ep_len.zero_()
        calls[0] += 1
        ep_len.add_(1)
        m.pass1(v, d["actions"], o, episode_length=ep_len)
        m.reset(origins, None, o, episode_length=ep_len)
        m.pass2(v, o)

    wl = ChainedWorkload(mdp, origins, out, PERIOD, 1234, cfg, stones_change=True, close_step=three_call)
    return wl


def time_steps(wl, steps: int) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        wl.step()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("envs", type=int, nargs="*", default=[65536, 1048576])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU and has nothing to report without one")
    print(f"card: {card()}", flush=True)
    for N in args.envs:
        wls = {B: make(N, B) for B in (0, 11)}
        for wl in wls.values():
            for _ in range(2 * PERIOD):
                wl.step()
        torch.cuda.synchronize()
        res = {0: [], 11: []}
        for _ in range(args.repeats):
            for B, wl in wls.items():
                res[B].append(time_steps(wl, args.steps))
        for B, wl in wls.items():
            s = wl.mdp.read_stats()
            ts = ", ".join(f"{t:.1f}" for t in res[B])
            print(f"N={N:>8}  grid {'11x11' if B else 'off  '}  us/step min {min(res[B]):8.1f}  (runs: {ts})  "
                  f"reset rate {100 * wl.reset_rate:.1f}%  regenerated last step {s['n_regenerated']}", flush=True)
        del wls
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
