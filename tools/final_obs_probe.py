"""Cost of AsStepOut.final_obs (the observation of the state an env's episode ended in, written for the envs that
reset): the fused step and the 3-call path with the device-side reset list, each with and without the output, on the
`workload.ChainedWorkload` cycle bench.py times (16 input sets, 2 % falls), at 1 048 576 and at 4096 envs.

The variants alternate inside one run (CUDA events around K steps, R rounds each); the card's name and power limit are
read in the same run.  Before timing, every step of one cycle is run twice from the same snapshot, with the output off
and on: all other outputs, the MDP state and the statistics must be bit-identical (the reward sum is accumulated by
float atomics in no fixed order and is reported as a difference).

    python tools/final_obs_probe.py [--steps K] [--rounds R] [--sizes 1048576,4096]

Prints one JSON line.  Writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--sizes", default="1048576,4096")
    args = ap.parse_args()

    import torch

    from allsteps_isaaclab_b200 import _cabi, build as _build

    if _cabi.LIB_PATH == _build.OUT and _build.is_stale():
        lib_dir = tempfile.TemporaryDirectory(prefix="allsteps_b200_")
        _cabi.LIB_PATH = _build.build(out=os.path.join(lib_dir.name, _cabi.LIB_NAME))
    from allsteps_isaaclab_b200 import synthetic as syn
    from allsteps_isaaclab_b200.config import AllstepsCfg
    from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers
    from allsteps_isaaclab_b200.workload import ChainedWorkload

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = AllstepsCfg()
    result = {"card": card(), "steps": args.steps, "rounds": args.rounds, "sizes": {}}

    for N in (int(s) for s in args.sizes.split(",")):
        seed = 1234
        origins = syn.env_origins_grid(N, cfg.env_spacing).to(dev)
        mdp = AllstepsMDP(N, device=dev, seed=seed)
        mdp.generate_stones(origins)
        st0 = syn.random_mdp_state(cfg, N, torch.Generator().manual_seed(seed))
        mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                              "episode_length_buf", "potentials")})
        off, on = StepBuffers(N, dev), StepBuffers(N, dev, final_obs=True)
        wl = ChainedWorkload(mdp, origins, off, 16, seed, cfg, 0.02)
        ep_len = torch.zeros(N, dtype=torch.int64, device=dev)

        def fused(v, d, out):
            mdp.step(v, d["actions"], out)

        def three_call(v, d, out):
            ep_len.add_(1)
            mdp.pass1(v, d["actions"], out, episode_length=ep_len)
            mdp.reset(origins, None, out, episode_length=ep_len)
            mdp.pass2(v, out)

        # ---- the outputs with the feature on and off, step by step from the same snapshot
        def outputs(out, compact_rows):
            d = {k: getattr(out, k).clone() for k in ("obs", "reward", "terminated", "time_out", "dones")}
            n = int(out.n_reset.item())
            order = out.reset_ids[:n].long().argsort()  # (the id list is filled by atomics: its order varies)
            ids = out.reset_ids[:n].long()[order]
            d["reset_ids"] = ids
            for k in ("reset_root_state", "reset_joint_pos", "reset_joint_vel"):
                t = getattr(out, k)
                d[k] = t[:n][order].clone() if compact_rows else t[ids].clone()
            d["state"] = mdp.export_state()
            d["stats"] = mdp.read_stats()
            return d

        def differences(a, b):
            bad = []
            for k in a:
                if k == "state":
                    bad += [f"state.{s}" for s in a[k] if not torch.equal(a[k][s].view(torch.uint8),
                                                                       b[k][s].view(torch.uint8))]
                elif k == "stats":
                    bad += [f"stats.{s}" for s in a[k] if s != "sum_reward" and a[k][s] != b[k][s]]
                elif not torch.equal(a[k].contiguous().view(torch.uint8), b[k].contiguous().view(torch.uint8)):
                    bad.append(k)
            return bad

        check = {}
        for name, fn, compact in (("fused", fused, False), ("three_call_device_list", three_call, True)):
            wl.rewind()
            bad, worst_sum, n_reset = set(), 0.0, 0
            for k in range(wl.period):
                v, d = wl.sets[k]
                snap, ep0 = mdp.snapshot(include_stones=False), ep_len.clone()
                fn(v, d, off)
                a = outputs(off, compact)
                mdp.restore(snap, include_stones=False)
                ep_len.copy_(ep0)
                on.final_obs.fill_(float("nan"))
                fn(v, d, on)
                b = outputs(on, compact)
                bad |= set(differences(a, b))
                worst_sum = max(worst_sum, abs(a["stats"]["sum_reward"] - b["stats"]["sum_reward"]))
                ids = b["reset_ids"]
                rows = on.final_obs[ids]
                others = torch.ones(N, dtype=torch.bool, device=dev)
                others[ids] = False
                if bool(rows.isnan().any()) or not bool(on.final_obs[others].isnan().all()):
                    bad.add("final_obs rows")  # written exactly for the envs that reset
                n_reset += len(ids)
            check[name] = {"other_outputs_state_stats_bit_identical": not bad, "differences": sorted(bad),
                           "sum_reward_max_abs_diff": worst_sum, "resets_in_cycle": n_reset,
                           "reset_rate": n_reset / (N * wl.period)}

        # ---- timing: the four variants alternate, R rounds of K steps each
        def timed(fn, out):
            wl.rewind()
            ep_len.zero_()
            for i in range(args.warmup):
                fn(*wl.sets[i % wl.period], out)
            wl.rewind()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                k = i % wl.period
                if k == 0 and i > 0:
                    wl.rewind()
                fn(*wl.sets[k], out)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e3 / args.steps  # us per step

        variants = [("fused", fused, off), ("fused+final_obs", fused, on),
                    ("three_call", three_call, off), ("three_call+final_obs", three_call, on)]
        times = {name: [] for name, _, _ in variants}
        for r in range(args.rounds):
            order = variants if r % 2 == 0 else variants[::-1]
            for name, fn, out in order:
                times[name].append(timed(fn, out))
        med = {k: statistics.median(v) for k, v in times.items()}
        result["sizes"][str(N)] = {
            "us_per_step_median": med,
            "us_per_step_all": times,
            "cost_us_fused": med["fused+final_obs"] - med["fused"],
            "cost_us_three_call": med["three_call+final_obs"] - med["three_call"],
            "spread_us_fused_off": max(times["fused"]) - min(times["fused"]),
            "spread_us_three_call_off": max(times["three_call"]) - min(times["three_call"]),
            "check": check,
        }
        del wl, mdp, off, on
        torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
