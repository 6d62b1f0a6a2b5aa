"""The global 3-call mode across shards against one handle holding all envs (run under torchrun, one rank per GPU).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/three_call_peer_check.py \
        [--num-steps S]

Every rank owns one env-id shard of the same seeded scenario and drives it through the 3-call path (`pass1` ->
`reset` -> `pass2`, or `no_reset`) in the global 3-call mode (`connect_peers(three_call=True)`); rank 0 also drives ONE
plain handle holding all envs through the same steps on the concatenated inputs.  At every step the shards' outputs
(obs, reward, masks, final observations, reset rows), state (levels and stones included) and grid bins must equal the
single handle's, their histograms must equal its histograms right after each pass 1, and the sums over the ranks of
the additive statistics must equal its statistics.  The scenario starts with a reset outside a step and then
alternates the host-id and the device-side-list route; it contains steps in which only one rank has falls -- there
the other ranks' `no_reset()` / empty-list `pass2` must keep pass 2 -- and steps without falls, and it must promote.
The tool asserts that it met each of these.  Then the same through `StandaloneAllstepsEnv(..., distributed=True)`.

THREE_CALL_CHECK_BACKEND=gloo runs the ranks as processes sharing GPU (rank % device_count), as tools/peer_check.py
does.  THREE_CALL_CHECK_MODE=local runs the shards shard-local (no peers: the 3-call path's behaviour before the
global mode) and reports the first step at which they part from the single handle, and what differs there.
--num-steps runs courses of S stones (default 20); the promotion threshold is scaled to 12 S / 20, so that the scenario
still promotes.
"""
import argparse
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import torch.distributed as dist

from allsteps_isaaclab_b200 import synthetic as syn
from allsteps_isaaclab_b200.config import AllstepsCfg
from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers
from allsteps_isaaclab_b200.sharding import STATS_ADDITIVE_FIELDS
from scenario import Scenario
from three_call_driver import OUTPUTS, reset_rows, three_call_step

STATE_KEYS = ("curr_target_index", "swing_leg", "target_reach_count", "episode_length_buf", "potentials")
# which ranks' envs may fall in step t (t % 4); the others get physics without falls or fast bodies
FALLS = ("all", "first", "last", "none")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--num-steps", type=int, default=20, help="stones per course (AllstepsCfg.num_steps)")
    S = ap.parse_args().num_steps
    cfg = AllstepsCfg(num_steps=S, curriculum_progress_threshold=AllstepsCfg().curriculum_progress_threshold * S / 20)
    lo = 9 * S // 20  # (indices from here up sit above the promotion threshold on average)
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    backend = os.environ.get("THREE_CALL_CHECK_BACKEND", "nccl")
    local = int(os.environ.get("LOCAL_RANK", rank)) if backend == "nccl" else rank % torch.cuda.device_count()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo")
    mode = os.environ.get("THREE_CALL_CHECK_MODE", "global")

    def gather_cat(t):
        """Every rank's tensor, concatenated in rank order, on the host."""
        src = t.contiguous() if backend == "nccl" else t.contiguous().cpu()
        parts = [torch.empty_like(src) for _ in range(world)]
        dist.all_gather(parts, src)
        return torch.cat(parts).cpu()

    per = int(os.environ.get("THREE_CALL_CHECK_ENVS", "1200"))
    steps = int(os.environ.get("THREE_CALL_CHECK_STEPS", "24"))
    B = int(os.environ.get("THREE_CALL_CHECK_GRID", "5"))
    N, seed = per * world, 29
    sc = Scenario(N, seed=seed, cfg=cfg)  # same seed on every rank: identical CPU-side scenario
    st0 = sc.initial_mdp_state()
    st0["curr_target_index"] = torch.randint(lo, S, (N,), generator=sc.gen)  # above the promotion threshold
    st0["episode_length_buf"] = torch.randint(0, 600, (N,), generator=sc.gen)  # no time-outs during the run
    sl = slice(rank * per, (rank + 1) * per)
    origins = sc.env_origins[sl].to(dev)
    shard = AllstepsMDP(per, device=dev, cfg=cfg, seed=seed, env_id_offset=rank * per, grid_bins=B)
    shard.generate_stones(origins)
    shard.import_state({k: st0[k][sl] for k in STATE_KEYS})
    if mode == "global":
        assert shard.connect_peers(three_call=True) == (world, rank)
    out = StepBuffers(per, dev, final_obs=True)
    ep = st0["episode_length_buf"][sl].to(dev)
    single = out_s = ep_s = None
    if rank == 0:
        single = AllstepsMDP(N, device=dev, cfg=cfg, seed=seed, grid_bins=B)
        single.generate_stones(sc.env_origins.to(dev))
        single.import_state({k: st0[k] for k in STATE_KEYS})
        out_s = StepBuffers(N, dev, final_obs=True)
        ep_s = st0["episode_length_buf"].to(dev)

    def physics(falls):
        st = shard.export_state(("steps_pos", "curr_target_index", "swing_leg"))
        full = [gather_cat(st[k]) for k in ("steps_pos", "curr_target_index", "swing_leg")]
        live = sc.physics(*full)
        calm = syn.random_physics_state(sc.cfg, *full, sc.gen, fall_fraction=0.0, fast_fraction=0.0)
        # (on the steep stones of hard grid bins the feet can sit high enough that the torso-to-feet height drops
        # below the level's termination height, ENV:401: a torso one metre up cannot fall)
        calm["root_pos_w"][:, 2] += 1.0
        calm["body_pos_w"][:, sc.body_indices[2], 2] += 1.0
        ranks = {"all": range(world), "first": [0], "last": [world - 1], "none": []}[falls]
        for r in range(world):
            if r not in ranks:
                for k in live:
                    live[k][r * per:(r + 1) * per] = calm[k][r * per:(r + 1) * per]
        return live

    def by_env(ids, rows, n):
        t = torch.zeros(n, rows.shape[1], device=rows.device)
        t[ids] = rows
        return t

    def compare(what):
        """Names of what differs between the shards (gathered) and the single handle; [] on ranks other than 0."""
        mine = {name: getattr(out, name) for name in OUTPUTS}
        mine["reset rows"] = by_env(ids, reset_rows(out, order), per)
        mine["episode_length"] = ep
        mine.update(shard.export_state())
        mine["bins"] = shard.grid_state()[0]
        got = {k: gather_cat(v.view(torch.uint8) if v.dtype == torch.bool else v) for k, v in mine.items()}
        if rank != 0:
            return []
        ref = {name: getattr(out_s, name) for name in OUTPUTS}
        ref["reset rows"] = by_env(ids_s, reset_rows(out_s, order_s), N)
        ref["episode_length"] = ep_s
        ref.update(single.export_state())
        ref["bins"] = single.grid_state()[0]
        return [k for k, v in ref.items()
                if not torch.equal(got[k], (v.view(torch.uint8) if v.dtype == torch.bool else v).cpu())]

    # ---- DirectRLEnv.reset() before the first step: a reset outside a step on every rank
    phys = physics("all")
    d = {k: v[sl].to(dev) for k, v in phys.items()}
    shard.reset(origins, torch.arange(per, device=dev), out, episode_length=ep)
    shard.pass2(PhysicsViews.from_dict(d, origins, sc.body_indices), out)
    ids, order = torch.arange(per, device=dev), torch.arange(per, device=dev)
    if rank == 0:
        dall = {k: v.to(dev) for k, v in phys.items()}
        single.reset(sc.env_origins.to(dev), torch.arange(N, device=dev), out_s, episode_length=ep_s)
        single.pass2(PhysicsViews.from_dict(dall, sc.env_origins.to(dev), sc.body_indices), out_s)
        ids_s, order_s = torch.arange(N, device=dev), torch.arange(N, device=dev)
    torch.cuda.synchronize()
    bad = compare("reset outside a step")
    assert not bad or mode == "local", f"reset outside a step: {bad} differ from the single handle"
    if bad and rank == 0:
        print(f"three_call_peer_check LOCAL DIFFERS at the reset outside a step: {', '.join(bad)}", flush=True)
    # the reset put every env back at index 1: indices above the promotion threshold again, so that steps promote
    high = {"curr_target_index": torch.randint(lo, S, (N,), generator=sc.gen)}
    shard.import_state({k: v[sl] for k, v in high.items()})
    if rank == 0:
        single.import_state(high)

    met = dict(one_rank_host=0, one_rank_list=0, none=0, host=0, device_list=0, promotions=0)
    level_before = int(gather_cat(shard.export_state(("curriculum",))["curriculum"]).max())
    first_bad = None
    for step in range(steps):
        falls = FALLS[step % 4]
        device_list = step % 2 == 1 if falls != "none" else (step // 4) % 2 == 1
        phys = physics(falls)
        d = {k: v[sl].to(dev) for k, v in phys.items()}
        views = PhysicsViews.from_dict(d, origins, sc.body_indices)
        hist = {}

        def after_pass1_shard():
            torch.cuda.synchronize()
            hist["shard"] = shard.grid_hist_tensor.clone()

        ids, order = three_call_step(shard, views, d, out, origins, ep, device_list, after_pass1_shard)
        flagged = gather_cat(out.dones.sum().reshape(1).to(torch.int64))  # per rank, as pass 1 flagged them
        if rank == 0:
            dall = {k: v.to(dev) for k, v in phys.items()}
            vall = PhysicsViews.from_dict(dall, sc.env_origins.to(dev), sc.body_indices)

            def after_pass1_single():
                torch.cuda.synchronize()
                hist["single"] = single.grid_hist_tensor.clone()

            ids_s, order_s = three_call_step(single, vall, dall, out_s, sc.env_origins.to(dev), ep_s, device_list,
                                             after_pass1_single)
        torch.cuda.synchronize()
        what = f"step {step} ({'device list' if device_list else 'host ids'}, flagged per rank {flagged.tolist()})"
        bad = compare(what)
        hists = gather_cat(hist["shard"].unsqueeze(0))
        if rank == 0 and not all(torch.equal(h, hist["single"].cpu()) for h in hists):
            bad.append("histograms after pass 1")
        sums = gather_cat(shard.stats_tensor[:STATS_ADDITIVE_FIELDS].clone().unsqueeze(0)).sum(0)
        if rank == 0 and not torch.equal(sums, single.stats_tensor[:STATS_ADDITIVE_FIELDS].cpu()):
            bad.append(f"summed statistics {sums.tolist()} vs {single.stats_tensor[:STATS_ADDITIVE_FIELDS].tolist()}")
        n_busy = int((flagged > 0).sum())
        kind = "none" if n_busy == 0 else ("one rank" if n_busy == 1 else "several ranks")
        if mode == "local":
            if rank == 0 and bad and first_bad is None:
                first_bad = step
                print(f"three_call_peer_check LOCAL DIFFERS first at {what}, {kind} reset: {', '.join(bad)}",
                      flush=True)
            continue
        if rank == 0:
            assert not bad, f"{what}: {bad} differ from the single handle"
        met["one_rank_host"] += kind == "one rank" and not device_list
        met["one_rank_list"] += kind == "one rank" and device_list
        met["none"] += kind == "none"
        met["device_list" if device_list else "host"] += 1
        level = int(gather_cat(shard.export_state(("curriculum",))["curriculum"]).max())
        met["promotions"] += level > level_before
        level_before = level
    if mode == "local":
        if rank == 0 and first_bad is None:
            print("three_call_peer_check LOCAL matched the single handle at every step", flush=True)
        dist.destroy_process_group()
        return
    assert all(v > 0 for v in met.values()), f"the scenario missed a case it must contain: {met}"
    assert shard.peer_status()["timeouts"] == 0
    standalone_env_check(rank, world, dev, gather_cat, cfg)
    if rank == 0:
        print(f"three_call_peer_check OK: world {world} ({backend}, grid {B}x{B}), {S} stones, {per} envs per rank, {steps} steps "
              f"+ a reset outside a step, shards == single handle; {met}", flush=True)
    dist.destroy_process_group()


def standalone_env_check(rank, world, dev, gather_cat, cfg):
    """`StandaloneAllstepsEnv(..., distributed=True)` on every rank against one plain env holding all envs (rank 0):
    reset() then steps through the hooks; observations, rewards, masks, levels and stones must be equal."""
    from allsteps_isaaclab_b200.env import StandaloneAllstepsEnv
    from test_gpu_faces import _fake_world, _install

    per, seed, B = 640, 37, 7
    N = per * world
    sc = Scenario(N, seed=seed, full_bodies=True, fall_fraction=0.08, cfg=cfg)
    sl = slice(rank * per, (rank + 1) * per)
    shard_sc = types.SimpleNamespace(N=per, joint_limits=sc.joint_limits, cfg=sc.cfg)

    def make(scn, phys, origins, **kw):
        robot, left, right = _fake_world(scn, phys)
        scene = types.SimpleNamespace(env_origins=origins.to(dev))
        return StandaloneAllstepsEnv(robot, left, right, scene, str(dev), sc.cfg, seed=seed, grid_bins=B, **kw)

    zero = sc.physics(torch.zeros(N, cfg.num_steps, 3), torch.ones(N, dtype=torch.int64), torch.zeros(N, dtype=torch.int64))
    env = make(shard_sc, {k: v[sl] for k, v in zero.items()}, sc.env_origins[sl], distributed=True)
    assert env.mdp.env_id_offset == rank * per
    ref = make(sc, zero, sc.env_origins) if rank == 0 else None
    busy = 0
    for step in range(-1, 10):
        st = env.mdp.export_state(("steps_pos", "curr_target_index", "swing_leg"))
        phys = sc.physics(*[gather_cat(st[k]) for k in ("steps_pos", "curr_target_index", "swing_leg")])
        _install(env.robot, env.sensor_left, env.sensor_right, {k: v[sl] for k, v in phys.items()})
        if ref is not None:
            _install(ref.robot, ref.sensor_left, ref.sensor_right, phys)
        if step < 0:  # DirectRLEnv.reset() on every rank
            res = (env.reset()[0]["policy"],)
            res_ref = (ref.reset()[0]["policy"],) if ref is not None else None
        else:
            obs, rew, term, to, _ = env.post_physics_step(phys["actions"][sl].to(dev))
            res = (obs["policy"], rew, term, to)
            if ref is not None:
                obs_r, rew_r, term_r, to_r, _ = ref.post_physics_step(phys["actions"].to(dev))
                res_ref = (obs_r["policy"], rew_r, term_r, to_r)
        torch.cuda.synchronize()
        got = [gather_cat(t.view(torch.uint8) if t.dtype == torch.bool else t) for t in res]
        state = {k: gather_cat(v) for k, v in env.mdp.export_state().items()}
        if ref is not None:
            for i, (g, r) in enumerate(zip(got, res_ref)):
                r = (r.view(torch.uint8) if r.dtype == torch.bool else r).cpu()
                assert torch.equal(g, r), f"standalone env step {step}: output {i} differs from the single env"
            for k, v in ref.mdp.export_state().items():
                assert torch.equal(state[k], v.cpu()), f"standalone env step {step}: state {k} differs"
            busy += step >= 0 and bool(got[2].any())
    if ref is not None:
        assert busy > 0


if __name__ == "__main__":
    main()
