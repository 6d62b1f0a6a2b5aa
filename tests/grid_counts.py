"""Test infrastructure: difficulty-grid histograms at the counts of a long run, and the grid formulas restated.

* `restated_*`: the docstring of oracle/grid_curriculum.py in plain Python ints -- the yardstick the oracle (and through
  it the kernels) is held to.
* `wrapping_weights`: the weight formula as the oracle and `grid_weight` computed it before they were made exact
  (uint64, the numerator wrapping past 2^64).  Kept to show that the histograms below tell the two apart.
* `crafted_histograms`: bins at 2^27 .. 2^32 - 1 attempts with 0 %, 50 % and 100 % success, and bins never played.
"""
from __future__ import annotations

from bisect import bisect_right
from itertools import accumulate

import numpy as np

U32_MAX = (1 << 32) - 1
LEVELS = (1 << 27, 1 << 28, (1 << 28) + (1 << 27), 1 << 31, U32_MAX)


def restated_weight(a: int, s: int) -> int:
    return 256 if a == 0 else 1 + (1024 * s * (a - s)) // (a * a + 1)


def restated_cdf(att, succ) -> list:
    return list(accumulate(restated_weight(int(a), int(s)) for a, s in zip(att, succ)))


def restated_sample(cdf: list, u24: int) -> int:
    return bisect_right(cdf, (int(u24) * cdf[-1]) >> 24)


def restated_fold(a: int, s: int, da: int, ds: int):
    if a + da > U32_MAX:
        a, s = a >> 1, s >> 1
    return a + da, s + ds


def wrapping_weights(att: np.ndarray, succ: np.ndarray) -> np.ndarray:
    a = att.astype(np.uint64)
    s = succ.astype(np.uint64)
    with np.errstate(over="ignore"):
        w = np.uint64(1) + (np.uint64(1024) * s * (a - s)) // (a * a + np.uint64(1))
    return np.where(a == 0, np.uint64(256), w).astype(np.uint32)


def crafted_histograms(B: int, seed: int):
    """(attempts, successes) as uint32 (B*B,): bin 0 at 2^28 attempts and 50 % success (the count at which the wrapping
    formula first fails), bin 1 never played, the others drawn from LEVELS x {0, a // 2, a} and the empty bin."""
    kinds = [(a, s) for a in LEVELS for s in (0, a // 2, a)] + [(0, 0)]
    rng = np.random.default_rng(seed)
    att = np.zeros(B * B, dtype=np.uint32)
    succ = np.zeros(B * B, dtype=np.uint32)
    for b in range(B * B):
        a, s = (1 << 28, 1 << 27) if b == 0 else (0, 0) if b == 1 else kinds[int(rng.integers(len(kinds)))]
        att[b], succ[b] = a, s
    return att, succ


def at_the_top(d_att: np.ndarray, seed: int):
    """Histograms that put every bin with outcomes this step right at the fold's threshold: attempts da - 1, da or
    da + 1 below 2^32 - 1 (so a + da = 2^32: halved; 2^32 - 1 and 2^32 - 2: added as they are), successes 0, a // 2
    or a.  Bins without outcomes sit at 2^32 - 1."""
    rng = np.random.default_rng(seed)
    att = np.full(d_att.shape[0], U32_MAX, dtype=np.uint32)
    succ = np.zeros(d_att.shape[0], dtype=np.uint32)
    k = 0
    for b, da in enumerate(d_att.tolist()):
        if da:
            a = U32_MAX - da + (1, 0, -1)[k % 3]
            att[b] = a
            succ[b] = (0, a // 2, a)[int(rng.integers(3))]
            k += 1
        else:
            succ[b] = (0, U32_MAX // 2, U32_MAX)[b % 3]
    return att, succ


# the GPU test's sampling scenario (tests/test_gpu_grid_counts.py), shared with the CPU check that it can fail
SAMPLING_ENVS, SAMPLING_SEED, SAMPLING_FALL = 8192, 23, 0.3
SAMPLING_GRIDS = (2, 11, 16)
