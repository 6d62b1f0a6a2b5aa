"""TEST INFRASTRUCTURE ONLY -- oracle of the pitch x yaw grid curriculum (EXTENSION, parity unpinned).

`BASELINE.json:north_star` asks for "adaptive pitch x yaw difficulty-grid curriculum sampling": a shared-memory
histogram of success over the difficulty grid and a warp-scan inverse-CDF sampler.  The reference has no such code
(its curriculum is one scalar level, SURVEY D2), so there is nothing to be bit-compatible with: this file IS the
specification, written first, and the CUDA kernels (csrc/as_grid_kernels.cuh) are checked against it bit for bit.
Everything that decides a bin is integer arithmetic, so "identical uniforms => identical bin" holds exactly.

Definition
  grid        B x B bins, bin b = i * B + j, i = pitch bin, j = yaw bin (B <= 16)
  difficulty  ratio_pitch = i / (B-1), ratio_yaw = j / (B-1) scale the +-30 deg / +-20 deg ranges of ENV:42-43 the way
              the scalar ratio does in ENV:131-132; dist upper bound = dist_upper[(max(i,j) * max_level) // (B-1)]
  outcome     an episode that ends (the env resets) is a success iff its curr_target_index had passed S/2
  histogram   two uint32 counters per bin: attempts (episodes ended in the bin) and successes (of those)
  fold        a step's outcomes join the histograms as one delta per bin, (da, ds) = episodes of the step that ended in
              the bin and how many of them were successes.  If a + da > 2^32 - 1 (in mathematical integers), the bin is
              halved first: (a, s) <- (a >> 1, s >> 1); then (a, s) <- (a + da, s + ds).  Halving keeps the success
              ratio and s <= a; a step's delta is at most the run's env count (< 2^31), so one halving makes room.  The
              rule depends on the global sums only, so shards keep identical histograms.  Below 2^32 - 1 - da it is a
              plain addition.
  precondition successes[b] <= attempts[b] for every bin, and every env's bin is < B * B
  weights     w_b = 256 if attempts == 0 else 1 + (1024 * s * (a - s)) // (a * a + 1)      (peaks at 50 % success)
              on mathematical integers (the numerator needs up to 72 bits).  With s <= a every weight is in 1..256,
              so the CDF total is at most 256 * 256 and fits a uint32 with room to spare.
  sampling    cdf = inclusive prefix sum of w; u24 = 24-bit uniform; target = (u24 * cdf[-1]) >> 24;
              new bin = first b with cdf[b] > target
  each env that resets is assigned a new bin and its stone sequence is regenerated at that bin's difficulty.
  order       bins drawn in step t come from the histograms as they stand after step t-1; the outcomes of step t are
              added afterwards.  (So that a run sharded over several GPUs can sum the step's outcomes over the ranks
              when it closes the step, off the sampling path, and still sample from exactly the CDF one handle holding
              all envs would use: the histograms are GLOBAL, every shard keeps an identical copy.)
"""
from __future__ import annotations

import numpy as np
import torch

from . import philox

STREAM_GRID = 2
U32_MAX = 0xFFFFFFFF  # the histogram counters are uint32


def weights(attempts: np.ndarray, successes: np.ndarray) -> np.ndarray:
    """The bin weights, evaluated in Python ints (exact; at most 256 bins)."""
    w = [256 if a == 0 else 1 + (1024 * s * (a - s)) // (a * a + 1)
         for a, s in zip(np.asarray(attempts).tolist(), np.asarray(successes).tolist())]
    return np.array(w, dtype=np.uint32)


def cdf_of(attempts: np.ndarray, successes: np.ndarray) -> np.ndarray:
    return np.cumsum(weights(attempts, successes).astype(np.uint64)).astype(np.uint32)


def sample_bins(cdf: np.ndarray, u24: np.ndarray) -> np.ndarray:
    total = np.uint64(cdf[-1])
    target = (u24.astype(np.uint64) * total) >> np.uint64(24)
    return np.searchsorted(cdf.astype(np.uint64), target, side="right").astype(np.uint8)


def fold(attempts: np.ndarray, successes: np.ndarray, d_att: np.ndarray, d_succ: np.ndarray) -> None:
    """A step's per-bin outcomes (d_att, d_succ) join the uint32 histograms in place (see "fold" above)."""
    for b, (da, ds) in enumerate(zip(np.asarray(d_att).tolist(), np.asarray(d_succ).tolist())):
        a, s = int(attempts[b]), int(successes[b])
        if a + da > U32_MAX:
            a, s = a >> 1, s >> 1
        attempts[b] = a + da
        successes[b] = s + ds


def grid_draws(seed: int, step: int, env_ids: np.ndarray) -> np.ndarray:
    """24-bit uniforms of stream 2, draw 0, for the envs being re-assigned."""
    env_ids = np.asarray(env_ids, dtype=np.uint32)
    n = env_ids.shape[0]
    counter = np.zeros((n, 4), dtype=np.uint32)
    counter[:, 0] = env_ids
    counter[:, 2] = np.uint32(step & 0xFFFFFFFF)
    counter[:, 3] = np.uint32(STREAM_GRID | (((step >> 32) & 0xFFFFFF) << 8))
    key = np.zeros((n, 2), dtype=np.uint32)
    key[:, 0] = np.uint32(seed & 0xFFFFFFFF)
    key[:, 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    return philox.philox4x32_10(counter, key)[:, 0] >> np.uint32(8)


def bin_difficulty(cfg, bins: torch.Tensor, B: int):
    """(ratio_yaw, ratio_pitch, dist_upper) per env for its bin."""
    i = (bins.long() // B).float()
    j = (bins.long() % B).float()
    denom = torch.tensor(float(B - 1))
    dist_table = torch.linspace(*torch.tensor(cfg.dist_range, dtype=torch.float32), cfg.max_curriculum + 1)
    k = (torch.maximum(bins.long() // B, bins.long() % B) * cfg.max_curriculum) // (B - 1)
    return j / denom, i / denom, dist_table[k]


def generate_stones_for_bins(cfg, bins: torch.Tensor, B: int, uniforms: torch.Tensor):
    """ENV:125-174 with the scalar `ratio` replaced by the per-axis ratios of each env's bin."""
    ratio_yaw, ratio_pitch, dist_hi = bin_difficulty(cfg, bins, B)
    N = bins.shape[0]
    yaw_lohi = torch.tensor(cfg.yaw_range_deg, dtype=torch.float32)
    pitch_lohi = torch.tensor(cfg.pitch_range_deg, dtype=torch.float32)
    dist_lo = torch.tensor(cfg.dist_range[0], dtype=torch.float32).repeat(N)
    yaw_range = torch.deg2rad(yaw_lohi.unsqueeze(0) * ratio_yaw.unsqueeze(1))
    pitch_range = torch.deg2rad(pitch_lohi.unsqueeze(0) * ratio_pitch.unsqueeze(1)) + torch.pi / 2
    dr = torch.lerp(dist_lo.unsqueeze(1), dist_hi.unsqueeze(1), uniforms[0])
    dphi = torch.lerp(yaw_range[:, 0].unsqueeze(1), yaw_range[:, 1].unsqueeze(1), uniforms[1])
    dtheta = torch.lerp(pitch_range[:, 0].unsqueeze(1), pitch_range[:, 1].unsqueeze(1), uniforms[2])
    dr[:, 0] = 0.0
    dphi[:, 0] = 0.0
    dtheta[:, 0] = torch.pi / 2
    dr[:, 1:3] = cfg.init_step_separation
    dphi[:, 1:3] = 0.0
    dtheta[:, 1:3] = torch.pi / 2
    dphi = torch.cumsum(dphi, dim=1)
    dx = dr * torch.sin(dtheta) * torch.cos(dphi)
    dy = dr * torch.sin(dtheta) * torch.sin(dphi)
    dz = dr * torch.cos(dtheta)
    pos = torch.stack((torch.cumsum(dx, 1), torch.cumsum(dy, 1), torch.cumsum(dz, 1)), dim=2)
    return pos, dphi


class GridCurriculum:
    """Host-side state of the extension: per-env bin and the two histograms."""

    def __init__(self, num_envs: int, B: int = 11, env_id_offset: int = 0):
        self.B = B
        self.bins = np.zeros(num_envs, dtype=np.uint8)
        self.attempts = np.zeros(B * B, dtype=np.uint32)
        self.successes = np.zeros(B * B, dtype=np.uint32)
        self.env_id_offset = env_id_offset

    def episode_end(self, env_ids: np.ndarray, index_at_end: np.ndarray, num_stones: int, seed: int, step: int):
        """Draw the new bins of the envs that reset from the histograms of the previous steps, then record this step's
        outcomes (see "order" above)."""
        b = self.bins[env_ids].copy()
        cdf = cdf_of(self.attempts, self.successes)
        u24 = grid_draws(seed, step, env_ids + self.env_id_offset)
        self.bins[env_ids] = sample_bins(cdf, u24)
        nb = self.attempts.shape[0]
        ok = np.asarray(index_at_end) > num_stones // 2
        fold(self.attempts, self.successes, np.bincount(b, minlength=nb), np.bincount(b[ok], minlength=nb))
        return self.bins[env_ids]
