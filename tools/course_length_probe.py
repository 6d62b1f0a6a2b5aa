"""Step times at other course lengths: the fused step and the 3-call path (pass1 -> reset on the device-side list ->
pass2) at 1 048 576 envs for S = 8, 20 and 32 stones (`AllstepsCfg.num_steps`), on the chained synthetic workload
bench.py times (allsteps_isaaclab_b200/workload.py).  S = 20 takes the FAST step-kernel instantiations, every other
length the generic ones, which read S from the parameters.

    python tools/course_length_probe.py [--envs 1048576] [--lengths 8 20 32] [--steps 200] [--warmup 20] [--out FILE]

Prints one JSON line per length (milliseconds per step, device time between CUDA events; the rewind at each cycle
start is inside) with the card's name and power limit read in the same run (`nvidia-smi --query-gpu`), and, with
--out, writes them to FILE.  Needs a B200; no CPU fallback.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from allsteps_isaaclab_b200 import synthetic as syn  # noqa: E402
from allsteps_isaaclab_b200.config import AllstepsCfg  # noqa: E402
from allsteps_isaaclab_b200.mdp import AllstepsMDP, StepBuffers  # noqa: E402
from allsteps_isaaclab_b200.workload import ChainedWorkload  # noqa: E402


def card(index=0):
    """(name, power limit) of the device the probe runs on, as nvidia-smi reports them (a read-only query)."""
    uuid = str(getattr(torch.cuda.get_device_properties(index), "uuid", ""))
    sel = ["-i", uuid if uuid.startswith("GPU-") else "GPU-" + uuid] if uuid else []
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", *sel],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, limit = (x.strip() for x in out[0].split(","))
        return name, limit
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(index), "unknown"


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def probe(S, n, steps, warmup, seed=1234, period=4):
    cfg = AllstepsCfg(num_steps=S)
    dev = torch.device("cuda:0")
    mdp = AllstepsMDP(n, device=dev, cfg=cfg, seed=seed)
    origins = syn.env_origins_grid(n, cfg.env_spacing).to(dev)
    mdp.generate_stones(origins)
    gen = torch.Generator().manual_seed(seed)
    st0 = syn.random_mdp_state(cfg, n, gen)
    mdp.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf",
                                          "potentials")})
    out = StepBuffers(n, dev)
    wl = ChainedWorkload(mdp, origins, out, period=period, seed=seed, cfg=cfg)
    fused = timed(wl.step, steps, warmup)
    ep_len = torch.zeros(n, dtype=torch.int64, device=dev)

    def three_call():
        k = wl.j % wl.period
        if k == 0 and wl.j > 0:
            wl.rewind()
        v, d = wl.sets[k]
        ep_len.add_(1)
        mdp.pass1(v, d["actions"], out, episode_length=ep_len)
        mdp.reset(origins, None, out, episode_length=ep_len)
        mdp.pass2(v, out)
        wl.j += 1

    wl.rewind()
    three = timed(three_call, steps, warmup)
    return {"num_steps": S, "envs": n, "fused_ms": round(fused, 4), "three_call_ms": round(three, 4),
            "advance_rate": round(wl.advance_rate, 4), "reset_rate": round(wl.reset_rate, 4)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--lengths", type=int, nargs="+", default=[8, 20, 32])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("course_length_probe needs a CUDA device (B200)")
    name, limit = card()
    rows = []
    for S in a.lengths:
        r = probe(S, a.envs, a.steps, a.warmup)
        r.update(gpu=name, power_limit=limit, steps=a.steps, warmup=a.warmup)
        print(json.dumps(r), flush=True)
        rows.append(r)
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()
