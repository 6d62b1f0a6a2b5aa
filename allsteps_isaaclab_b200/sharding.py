"""Env-id sharding over the GPUs of one box (SURVEY section 8e).

Every env is independent on the step path, so the N global envs are cut into contiguous id ranges, one per rank
(one process per GPU, `torchrun`).  Philox draws are keyed by GLOBAL env id (`AllstepsMDP(env_id_offset=...)`), so
results do not depend on the number of ranks.  Nothing is exchanged on the step path; the only cross-env quantities
are the step statistics (numerator/denominator of the promotion rule ENV:471, episode counters), summed with one
small all-reduce -- NCCL on the GPUs, gloo in the CPU tests.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from ._cabi import EXCHANGE_INT64_WORDS, STATS_ADDITIVE_FIELDS, STATS_INT64_WORDS, AsStats

STAT_NAMES = [name for name, _ in AsStats._fields_]
SHARD_ALIGN = 4  # rows: keeps every shard's tiles 16-byte aligned for the TMA bulk copies


def shard_range(global_envs: int, rank: int, world: int, align: int = SHARD_ALIGN) -> Tuple[int, int]:
    """[start, stop) of `rank`'s contiguous env ids; shard starts are multiples of `align`."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    per = -(-global_envs // world)  # ceil
    per = -(-per // align) * align
    start = min(rank * per, global_envs)
    stop = min(start + per, global_envs)
    return start, stop


def global_env_offset(num_envs: int, device, group=None) -> int:
    """This rank's first global env id: the exclusive prefix sum of every rank's `num_envs` (one all_gather; on the
    GPU for NCCL, on the host for gloo).  Shards may differ in size; ids follow rank order."""
    import torch.distributed as dist

    dev = torch.device(device) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    mine = torch.tensor([int(num_envs)], dtype=torch.int64, device=dev)
    every = [torch.empty_like(mine) for _ in range(dist.get_world_size(group))]
    dist.all_gather(every, mine, group=group)
    return int(sum(int(t.item()) for t in every[:dist.get_rank(group)]))


def all_reduce_exchange(buf: torch.Tensor, with_grid: bool, group=None) -> torch.Tensor:
    """Sum an `AsExchange` record (int64 view: `AllstepsMDP.exchange_tensor` copied after `fold_stats()`) over the ranks
    where it is additive: the ten leading step counters and -- `with_grid` -- the step's difficulty-grid outcomes (two
    uint32 counters per int64 word; counts of one step cannot carry from the low half into the high one).  Level, step
    counter, reward sum and the missed-step counter stay this shard's.  NCCL on the GPUs, gloo in the CPU tests."""
    import torch.distributed as dist

    if buf.numel() < EXCHANGE_INT64_WORDS or buf.dtype != torch.int64:
        raise ValueError(f"an exchange record is {EXCHANGE_INT64_WORDS} int64 words")
    dist.all_reduce(buf[:STATS_ADDITIVE_FIELDS], group=group)
    if with_grid:
        dist.all_reduce(buf[STATS_INT64_WORDS:EXCHANGE_INT64_WORDS], group=group)
    return buf


class StatsReducer:
    """Sums the additive head of `AsStats` over ranks (async, off the step path) and applies the promotion rule."""

    def __init__(self, device, process_group=None, threshold: float = 12.0):
        self.device = torch.device(device)
        self.group = process_group
        self.threshold = threshold
        self.buf = torch.zeros(STATS_ADDITIVE_FIELDS, dtype=torch.int64, device=self.device)
        self.work = None

    def start(self, local_stats: torch.Tensor):
        """`local_stats`: int64 view of the device `AsStats` (AllstepsMDP.stats_tensor) or a CPU tensor."""
        import torch.distributed as dist

        self.buf.copy_(local_stats[:STATS_ADDITIVE_FIELDS])
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            self.work = dist.all_reduce(self.buf, group=self.group, async_op=True)
        return self

    def wait(self) -> Dict[str, int]:
        if self.work is not None:
            self.work.wait()
            self.work = None
        vals = self.buf.tolist()
        return dict(zip(STAT_NAMES[:STATS_ADDITIVE_FIELDS], vals))

    def promotes(self, stats: Optional[Dict[str, int]] = None) -> bool:
        """ENV:471-472 on the summed statistics: any reset and mean(curr_target_index) > threshold, in fp32."""
        s = stats or self.wait()
        if s["n_reset"] <= 0 or s["n_envs"] <= 0:
            return False
        mean = torch.tensor(float(s["sum_target_index"]), dtype=torch.float32) / torch.tensor(
            float(s["n_envs"]), dtype=torch.float32)
        return bool(mean > self.threshold)
