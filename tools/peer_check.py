"""Cross-shard promotion over NVLink peer memory against the NCCL route (run under torchrun, one rank per GPU).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/peer_check.py

Every rank owns one env-id shard of the same seeded scenario and steps it twice per step: once closing the step with
as_fold_stats -> all-reduce -> as_finish_step(global) and once with the peer-memory exchange kernel
(AllstepsMDP.connect_peers).  Outputs, MDP state and levels must be bit-identical between the two on every rank, the
global counters must equal the all-reduced sum, promotions must actually occur, and rank 0 also steps ONE handle
holding all envs: every rank's shard must equal its slice of that single handle.  Then the routes are timed.

PEER_CHECK_BACKEND=gloo runs the ranks as processes sharing GPU (rank % device_count) -- CUDA IPC peer memory works
between processes on one device too -- with the all-reduce going through gloo on host copies: the same check on a
one-GPU box.  PEER_CHECK_MODE=timeout: rank 1 connects but never steps; rank 0's exchange must time out, close the
step on its own counters and make every later step fail with AS_ERR_PEER.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import torch.distributed as dist

from allsteps_isaaclab_b200.mdp import AllstepsMDP, PhysicsViews, StepBuffers
from scenario import Scenario


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    backend = os.environ.get("PEER_CHECK_BACKEND", "nccl")
    if backend == "gloo":
        local = rank % torch.cuda.device_count()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo")

    def all_reduce(t, op=dist.ReduceOp.SUM):
        if backend == "nccl":
            dist.all_reduce(t, op=op)
        else:
            c = t.cpu()
            dist.all_reduce(c, op=op)
            t.copy_(c)

    def all_gather_cat(t):
        src = t.contiguous() if backend == "nccl" else t.contiguous().cpu()
        parts = [torch.empty_like(src) for _ in range(world)]
        dist.all_gather(parts, src)
        return torch.cat(parts).cpu()

    if os.environ.get("PEER_CHECK_MODE") == "timeout":
        return timeout_mode(rank, world, dev)
    per = int(os.environ.get("PEER_CHECK_ENVS", "4096"))
    steps = int(os.environ.get("PEER_CHECK_STEPS", "24"))
    N, seed = per * world, 17
    sc = Scenario(N, seed=seed)                     # same seed on every rank: identical CPU-side scenario
    st0 = sc.initial_mdp_state()
    st0["curr_target_index"] = torch.randint(11, 20, (N,), generator=sc.gen)   # near the promotion threshold
    sl = slice(rank * per, (rank + 1) * per)
    origins = sc.env_origins[sl].to(dev)
    grid = int(os.environ.get("PEER_CHECK_GRID", "0"))  # B > 0: pitch x yaw grid curriculum with global histograms
    mdps = [AllstepsMDP(per, device=dev, seed=seed, env_id_offset=rank * per, grid_bins=grid) for _ in range(2)]
    for m in mdps:
        m.generate_stones(origins)
        m.import_state({k: st0[k][sl] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                                "episode_length_buf", "potentials")})
    nccl_mdp, peer_mdp = mdps
    assert peer_mdp.connect_peers() == (world, rank)
    # PEER_CHECK_NEAR_TOP=1 (with a grid): every handle starts from histograms a few counts below 2^32 - 1, so the
    # steps' global outcomes halve bins (the fold of oracle/grid_curriculum.py) -- the same bins on every shard
    near_top = grid and os.environ.get("PEER_CHECK_NEAR_TOP") == "1"
    if near_top:
        nb = grid * grid
        top = torch.tensor([(1 << 32) - 1 - (b % 64) for b in range(nb)], dtype=torch.int64)
        hist0 = (top, top * (torch.arange(nb) % 3) // 2)
        for m in mdps:
            m.set_grid_state(None, *hist0)
    single = None
    if rank == 0:  # ONE handle with all envs: what every shard has to reproduce
        single = AllstepsMDP(N, device=dev, seed=seed, grid_bins=grid)
        single.generate_stones(sc.env_origins.to(dev))
        single.import_state({k: st0[k] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                                 "episode_length_buf", "potentials")})
        if near_top:
            single.set_grid_state(None, *hist0)
        out_single = StepBuffers(N, dev)
    outs = [StepBuffers(per, dev), StepBuffers(per, dev)]
    g = torch.zeros_like(nccl_mdp.exchange_tensor)

    def reduce_record(buf):
        all_reduce(buf[:10])
        if grid:
            all_reduce(buf[nccl_mdp.grid_words])
        return buf

    promotions = 0
    level_before = 0
    for step in range(steps):
        st = nccl_mdp.export_state()
        # the scenario needs the stones / indices of ALL envs: gather the shards
        full = {k: all_gather_cat(st[k]) for k in ("steps_pos", "curr_target_index", "swing_leg")}
        phys = sc.physics(full["steps_pos"], full["curr_target_index"], full["swing_leg"])
        d = {k: v[sl].to(dev) for k, v in phys.items()}
        views = PhysicsViews.from_dict(d, origins, sc.body_indices)
        nccl_mdp.step(views, d["actions"], outs[0], finish=False)
        nccl_mdp.fold_stats()
        g.copy_(nccl_mdp.exchange_tensor)
        nccl_mdp.finish_step(reduce_record(g))
        peer_mdp.step(views, d["actions"], outs[1])
        torch.cuda.synchronize()
        if single is not None:
            dall = {k: v.to(dev) for k, v in phys.items()}
            single.step(PhysicsViews.from_dict(dall, sc.env_origins.to(dev), sc.body_indices), dall["actions"],
                        out_single)
            torch.cuda.synchronize()
        # every rank's shard against its slice of the single handle (rank 0 broadcasts the whole result)
        for name in ("obs", "reward", "terminated", "time_out"):
            mine = getattr(outs[1], name)
            shape = (N,) + tuple(mine.shape[1:])
            whole = getattr(out_single, name) if rank == 0 else torch.empty(shape, dtype=mine.dtype, device=dev)
            whole = whole.view(torch.uint8) if whole.dtype == torch.bool else whole
            if backend == "nccl":
                dist.broadcast(whole, src=0)
                whole = whole.cpu()
            else:
                whole = whole.cpu()
                dist.broadcast(whole, src=0)
            ref = whole[sl]
            got = mine.view(torch.uint8).cpu() if mine.dtype == torch.bool else mine.cpu()
            assert torch.equal(got, ref), f"rank {rank} step {step}: {name} differs from the single handle"
        for name in ("obs", "reward", "terminated", "time_out", "dones", "reset_joint_pos"):
            a, b = getattr(outs[0], name), getattr(outs[1], name)
            assert torch.equal(a, b), f"rank {rank} step {step}: {name} differs between the NCCL and the peer route"
        sa, sb = nccl_mdp.export_state(), peer_mdp.export_state()
        for k in sa:
            assert torch.equal(sa[k], sb[k]), f"rank {rank} step {step}: state {k}"
        assert torch.equal(peer_mdp.global_stats_tensor[:10], g[:10]), (
            f"rank {rank} step {step}: global counters {peer_mdp.global_stats_tensor[:10].tolist()} vs NCCL "
            f"{g[:10].tolist()}")
        if grid:  # every shard holds the histograms of ALL envs: equal between the routes and to the single handle's
            ga, gb = nccl_mdp.grid_state(), peer_mdp.grid_state()
            assert torch.equal(ga[1], gb[1]) and torch.equal(ga[2], gb[2]) and torch.equal(ga[0], gb[0]), (
                f"rank {rank} step {step}: grid state differs between the routes")
            hist = torch.stack((gb[1], gb[2])).cpu()
            if backend == "nccl":
                h0 = hist.to(dev)
                dist.broadcast(h0, src=0)
                h0 = h0.cpu()
            else:
                h0 = hist.clone()
                dist.broadcast(h0, src=0)
            assert torch.equal(hist, h0), f"rank {rank} step {step}: histograms differ between the ranks"
            if single is not None:
                gs = single.grid_state()
                assert torch.equal(gs[1], gb[1]) and torch.equal(gs[2], gb[2]), "histograms differ from the single handle's"
                assert torch.equal(gs[0][sl], gb[0]), "bins differ from the single handle's"
                assert int(gs[1].sum()) > 0 or step == 0
        level = int(sb["curriculum"].max())
        promotions += int(level != level_before or grid > 0)
        level_before = level
    if near_top:
        att_end = peer_mdp.grid_state()[1].cpu()
        assert bool((att_end < hist0[0] // 2 + (1 << 20)).any()), "no bin was halved; the check would prove nothing"
    status = peer_mdp.peer_status()
    assert status["timeouts"] == 0 and status["world"] == world, status
    assert promotions > 0, "no promotion happened; the check would prove nothing"

    # ---- timing of the three ways to close a step (device time, max over ranks)
    def timed(fn, reps=200):
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps * 1e3], device=dev)
        all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    local_mdp = AllstepsMDP(per, device=dev, seed=seed, env_id_offset=rank * per, grid_bins=grid)
    local_mdp.generate_stones(origins)
    out_l = StepBuffers(per, dev)

    def via_nccl():
        nccl_mdp.step(views, d["actions"], outs[0], finish=False)
        nccl_mdp.fold_stats()
        g.copy_(nccl_mdp.exchange_tensor)
        nccl_mdp.finish_step(reduce_record(g))

    t_local = timed(lambda: local_mdp.step(views, d["actions"], out_l))
    t_nccl = timed(via_nccl)
    t_peer = timed(lambda: peer_mdp.step(views, d["actions"], outs[1]))
    assert peer_mdp.peer_status()["timeouts"] == 0
    if rank == 0:
        print(f"peer_check OK: world {world} ({backend}{', grid %dx%d' % (grid, grid) if grid else ''}"
              f"{' near the top of the counters' if near_top else ''}), {per} envs per rank, {steps} steps, {promotions} promotions, "
              f"shards == single handle; us/step: shard-local {t_local:.1f}, {backend} all-reduce {t_nccl:.1f}, "
              f"peer-memory exchange {t_peer:.1f}", flush=True)
    dist.destroy_process_group()


def timeout_mode(rank, world, dev):
    """Rank 1 connects and then stays away; rank 0 must not hang, must not use a partial sum, and must refuse to go on."""
    from allsteps_isaaclab_b200._cabi import AllstepsLibraryError

    per, seed = 2048, 5
    sc = Scenario(per * world, seed=seed)
    sl = slice(rank * per, (rank + 1) * per)
    origins = sc.env_origins[sl].to(dev)
    st0 = sc.initial_mdp_state()
    mdp = AllstepsMDP(per, device=dev, seed=seed, env_id_offset=rank * per)
    mdp.generate_stones(origins)
    mdp.import_state({k: st0[k][sl] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                              "episode_length_buf", "potentials")})
    mdp.connect_peers()
    if rank == 0:
        twin = AllstepsMDP(per, device=dev, seed=seed, env_id_offset=0)   # same shard, shard-local promotion
        twin.generate_stones(origins)
        twin.import_state({k: st0[k][sl] for k in ("curr_target_index", "swing_leg", "target_reach_count",
                                                   "episode_length_buf", "potentials")})
        st = mdp.export_state()
        phys = sc.physics(torch.cat([st["steps_pos"].cpu()] * world), torch.cat([st["curr_target_index"].cpu()] * world),
                          torch.cat([st["swing_leg"].cpu()] * world))
        d = {k: v[sl].to(dev) for k, v in phys.items()}
        views = PhysicsViews.from_dict(d, origins, sc.body_indices)
        out, out_t = StepBuffers(per, dev), StepBuffers(per, dev)
        mdp.step(views, d["actions"], out)        # the exchange waits ALLSTEPS_PEER_TIMEOUT_MS, then gives up
        twin.step(views, d["actions"], out_t)
        torch.cuda.synchronize()
        assert torch.equal(out.obs, out_t.obs), "the timed-out step must close on the shard's own counters"
        a, b = mdp.export_state(), twin.export_state()
        for k in a:
            assert torch.equal(a[k], b[k]), k
        assert mdp.peer_status()["timeouts"] >= 1
        try:
            mdp.step(views, d["actions"], out)
            raise SystemExit("a step after a peer timeout must fail")
        except AllstepsLibraryError as e:
            assert "(-4)" in str(e) and "timed out" in str(e), str(e)
        print("peer_check timeout OK: the exchange gave up, the step closed shard-locally, later steps are refused",
              flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
