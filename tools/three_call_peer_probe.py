"""Device time of one sharded env step on the 3-call path (as_step_pass1 -> as_reset -> as_step_pass2 / as_step_no_reset,
what the Isaac Lab faces drive), shard-local against the global 3-call mode (`connect_peers(three_call=True)`: one
peer-memory exchange behind every pass 1), with host ids (`dones.nonzero()`, the DirectRLEnv hooks) and with the
device-side list (`reset(None)`), on the chained synthetic workload (development tool, not the bench).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G tools/three_call_peer_probe.py [N ...] [--steps K]

N: envs per rank (default 131072 and 1048576).  One rank per GPU; with fewer GPUs than ranks, ranks share GPUs
(rank % device count), which times the sharing, not the exchange.  Rank 0 prints every card's name and power limit
first: a time belongs to the cards it was measured on.  Each configuration is timed R times, shard-local and global
alternating, with CUDA events around K steps after a barrier; the figure is the slowest rank's.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from allsteps_isaaclab_b200 import synthetic as syn  # noqa: E402
from allsteps_isaaclab_b200.config import AllstepsCfg  # noqa: E402
from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers  # noqa: E402
from allsteps_isaaclab_b200.workload import ChainedWorkload  # noqa: E402

PERIOD = 8


def cards() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or torch.cuda.get_device_name(0)
    except (OSError, subprocess.TimeoutExpired):
        return f"{torch.cuda.get_device_name(0)} (power limit not readable)"


def make(N, rank, dev, global_mode, device_list):
    cfg = AllstepsCfg()
    origins = syn.env_origins_grid(N, cfg.env_spacing).to(dev)
    mdp = AllstepsMDP(N, device=dev, seed=1, env_id_offset=rank * N, grid_bins=11)
    if global_mode:
        mdp.connect_peers(three_call=True)
    mdp.generate_stones(origins)
    st0 = syn.random_mdp_state(cfg, N, torch.Generator().manual_seed(1 + rank))
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
        if device_list:
            m.reset(origins, None, o, episode_length=ep_len)
            m.pass2(v, o)
            return
        ids = o.dones.nonzero().squeeze(-1)  # DRL:359 (a host round trip, as in the hooks)
        if len(ids):
            m.reset(origins, ids, o, episode_length=ep_len)
            m.pass2(v, o)
        else:
            m.no_reset()

    return ChainedWorkload(mdp, origins, out, PERIOD, 1234 + rank, cfg, stones_change=True, close_step=three_call)


def time_steps(wl, steps, dev) -> float:
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        wl.step()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([1e3 * e0.elapsed_time(e1) / steps], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("envs", type=int, nargs="*", default=[131072, 1048576])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this probe measures the GPU and has nothing to report without one")
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo")  # (the probe's own barriers and maxima; the step path uses no collective)
    if rank == 0:
        print(f"cards:\n{cards()}\nworld {world}, {torch.cuda.device_count()} GPU(s) visible", flush=True)
    for N in args.envs:
        for device_list in (False, True):
            wls = {g: make(N, rank, dev, g, device_list) for g in (False, True)}
            for wl in wls.values():
                for _ in range(2 * PERIOD):
                    wl.step()
            res = {False: [], True: []}
            for _ in range(args.repeats):
                for g, wl in wls.items():
                    res[g].append(time_steps(wl, args.steps, dev))
            if rank == 0:
                route = "device list" if device_list else "host ids   "
                lo, gl = min(res[False]), min(res[True])
                print(f"N/rank={N:>8}  {route}  us/step min: shard-local {lo:8.1f}  global {gl:8.1f}  "
                      f"(+{gl - lo:.1f})  runs local {[round(t, 1) for t in res[False]]} "
                      f"global {[round(t, 1) for t in res[True]]}  reset rate {100 * wls[True].reset_rate:.1f}%",
                      flush=True)
            del wls
            torch.cuda.empty_cache()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
