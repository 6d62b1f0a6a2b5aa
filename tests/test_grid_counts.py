"""CPU: the grid curriculum's specification (oracle/grid_curriculum.py) at the histogram counts of a long run, against
its own docstring restated in plain Python ints (tests/grid_counts.py): the weights, the CDF and the inverse-CDF
search over the whole uint32 range of the counters, and the fold that keeps them from wrapping."""
from __future__ import annotations

import numpy as np
import pytest

from grid_counts import (LEVELS, SAMPLING_ENVS, SAMPLING_GRIDS, SAMPLING_SEED, U32_MAX, crafted_histograms,
                         restated_cdf, restated_fold, restated_sample, restated_weight, wrapping_weights)
from oracle import grid_curriculum as gc


def _structured_pairs():
    edges = set(range(4)) | {2 ** k + d for k in range(8, 32) for d in (-1, 0, 1)} | {U32_MAX}
    pairs = []
    for a in sorted(edges):
        for s in sorted({0, 1, a // 2 - 1, a // 2, a // 2 + 1, a - 1, a}):
            if 0 <= s <= a:
                pairs.append((a, s))
    return pairs


def _random_pairs(n, seed):
    rng = np.random.default_rng(seed)
    a = np.minimum(np.floor(2.0 ** rng.uniform(0.0, 32.0, n)).astype(np.uint64), np.uint64(U32_MAX))
    s = np.floor(rng.uniform(0.0, 1.0, n) * (a.astype(np.float64) + 1.0)).astype(np.uint64)
    return list(zip(a.tolist(), np.minimum(s, a).tolist()))


@pytest.mark.parametrize("pairs", ["structured", "random"])
def test_weights_are_exact_over_the_whole_counter_range(pairs):
    """The numerator 1024 * s * (a - s) needs up to 72 bits: from s * (a - s) >= 2^54 (about 2^28 attempts at 50 %
    success) a 64-bit product wraps and the bins the curriculum wants most drop to weight 1."""
    pairs = _structured_pairs() if pairs == "structured" else _random_pairs(100_000, 5)
    att = np.array([a for a, _ in pairs], dtype=np.uint32)
    succ = np.array([s for _, s in pairs], dtype=np.uint32)
    got = gc.weights(att, succ)
    assert got.dtype == np.uint32 and got.shape == att.shape
    want = np.array([restated_weight(a, s) for a, s in pairs], dtype=np.int64)
    bad = np.nonzero(got.astype(np.int64) != want)[0]
    assert bad.size == 0, (f"{bad.size} of {len(pairs)} weights differ, first (a, s) = {pairs[bad[0]]}: "
                           f"{int(got[bad[0]])} vs {int(want[bad[0]])}")
    assert want.min() >= 1 and want.max() <= 256
    # the rows of the table in oracle/grid_curriculum.py's history: 50 % bins weigh 256 at every count
    for a in (1 << 27, 1 << 28, 3 << 27, 1 << 31, U32_MAX):
        assert int(gc.weights(np.array([a], np.uint32), np.array([(a + 1) // 2], np.uint32))[0]) == 256, a


def _valid_histograms():
    rng = np.random.default_rng(11)
    yield np.full(256, U32_MAX, np.uint32), np.full(256, U32_MAX // 2, np.uint32)  # every bin at the top, 50 %
    yield np.full(256, U32_MAX, np.uint32), np.full(256, U32_MAX, np.uint32)
    yield np.zeros(256, np.uint32), np.zeros(256, np.uint32)
    for B in (2, 5, 11, 16):
        yield crafted_histograms(B, B)
    for _ in range(50):
        nb = int(rng.integers(1, 257))
        a = np.array([int(2.0 ** x) if x > 0.5 else 0 for x in rng.uniform(0.0, 32.0, nb)], dtype=np.uint64)
        a = np.minimum(a, U32_MAX)
        s = np.minimum(np.floor(rng.uniform(0, 1, nb) * (a.astype(np.float64) + 1)).astype(np.uint64), a)
        yield a.astype(np.uint32), s.astype(np.uint32)


def test_cdf_is_monotone_and_bounded_for_any_valid_histogram():
    for att, succ in _valid_histograms():
        cdf = gc.cdf_of(att, succ)
        assert cdf.dtype == np.uint32
        c = cdf.astype(np.int64)
        assert np.all(np.diff(c) >= 1), "every bin has a positive weight"
        assert 1 <= c[0] and c[-1] <= 256 * 257
        assert c.tolist() == restated_cdf(att.tolist(), succ.tolist())


def _crossings(cdf):
    """u24 values where target = (u24 * total) >> 24 first reaches each cdf[b], and the value just below."""
    total = int(cdf[-1])
    us = {0, (1 << 24) - 1}
    for c in cdf.tolist():
        u = -(-(c << 24) // total)  # smallest u with u * total >= c * 2^24
        us |= {x for x in (u - 1, u, u + 1) if 0 <= x < 1 << 24}
    return np.array(sorted(us), dtype=np.uint32)


@pytest.mark.parametrize("case", ["crafted", "zero_width"])
def test_sample_bins_at_every_crossing(case):
    """Inverse-CDF search at 0, 2^24 - 1 and both sides of every bin edge; a bin of zero width is never drawn."""
    if case == "crafted":
        cdfs = [gc.cdf_of(*crafted_histograms(B, B)) for B in (2, 11, 16)]
        cdfs.append(gc.cdf_of(np.full(256, U32_MAX, np.uint32), np.full(256, U32_MAX // 2, np.uint32)))
    else:  # sample_bins takes any non-decreasing CDF: repeated values are bins of weight 0
        cdfs = [np.array([0, 5, 5, 9, 9, 9, 12, 12], np.uint32), np.array([0, 0, 1], np.uint32),
                np.array([3, 3, 3, 65536, 65536], np.uint32)]
    for cdf in cdfs:
        u24 = _crossings(cdf)
        got = gc.sample_bins(cdf, u24)
        c = cdf.tolist()
        want = [restated_sample(c, u) for u in u24.tolist()]
        assert got.tolist() == want
        width = np.diff(np.concatenate(([0], cdf.astype(np.int64))))
        assert np.all(width[got.astype(np.int64)] > 0), "a bin of zero width was drawn"
        assert got.max() < len(c)


def test_fold_halves_a_bin_only_when_its_attempts_would_pass_the_counter():
    for da in (1, 2, 7, 1 << 20, (1 << 31) - 1):
        for a in (U32_MAX - da, U32_MAX - da + 1, U32_MAX):
            for s in sorted({0, 1, a // 2, a - 1, a}):
                for ds in sorted({0, da // 2, da}):
                    att = np.array([a], np.uint32)
                    succ = np.array([s], np.uint32)
                    gc.fold(att, succ, np.array([da]), np.array([ds]))
                    want = restated_fold(a, s, da, ds)
                    assert (int(att[0]), int(succ[0])) == want, (a, s, da, ds)
                    assert int(succ[0]) <= int(att[0])
                    assert (want[0] == a + da) == (a + da <= U32_MAX)  # a plain addition up to the top


def test_episode_end_draws_from_the_old_histograms_then_folds():
    """GridCurriculum.episode_end (and ThreeCallGrid, which inherits it) against the restatement: bins from the CDF as
    the histograms stood, then one delta per bin, folded."""
    rng = np.random.default_rng(3)
    for B, N, seed, step in ((2, 500, 1, 0), (11, 3000, 2, 7), (16, 4000, 3, 1 << 33)):
        nb = B * B
        g = gc.GridCurriculum(N, B, env_id_offset=17)
        g.bins[:] = rng.integers(0, nb, N)
        ids = np.sort(rng.choice(N, N // 3, replace=False))
        played = g.bins[ids].astype(np.int64)
        da = np.bincount(played, minlength=nb)
        # every bin with outcomes at the fold's threshold, or one either side
        att = np.array([min(U32_MAX, U32_MAX - int(d) + (1, 0, -1)[b % 3]) for b, d in enumerate(da)], np.uint32)
        succ = np.array([(0, int(a) // 2, int(a))[b % 3] for b, a in enumerate(att)], np.uint32)
        g.attempts[:], g.successes[:] = att, succ
        index_at_end = rng.integers(0, 21, ids.size)
        cdf = restated_cdf(att.tolist(), succ.tolist())
        u24 = gc.grid_draws(seed, step, ids + 17)
        got = g.episode_end(ids, index_at_end, 20, seed, step)
        assert got.tolist() == [restated_sample(cdf, u) for u in u24.tolist()]
        ds = np.bincount(played[index_at_end > 10], minlength=nb)
        want = [restated_fold(int(a), int(s), int(x), int(y)) for a, s, x, y in zip(att, succ, da, ds)]
        assert g.attempts.tolist() == [w[0] for w in want] and g.successes.tolist() == [w[1] for w in want]
        assert np.all(g.successes <= g.attempts)
        assert any(w[0] < a for w, a in zip(want, att.tolist())), "no bin was halved"


@pytest.mark.parametrize("B", SAMPLING_GRIDS)
def test_wrapping_weights_draw_other_bins_on_the_gpu_tests_histograms(B):
    """The GPU test of the sampler at large counts can fail: on its histograms the formula with the 64-bit wrap gives
    other bins than the exact one for many envs."""
    att, succ = crafted_histograms(B, SAMPLING_SEED + B)
    assert max(att.tolist()) in LEVELS
    u24 = gc.grid_draws(SAMPLING_SEED, 0, np.arange(SAMPLING_ENVS))
    exact_bins = gc.sample_bins(gc.cdf_of(att, succ), u24)
    wrapping = gc.sample_bins(np.cumsum(wrapping_weights(att, succ).astype(np.uint64)).astype(np.uint32), u24)
    assert int((exact_bins != wrapping).sum()) > SAMPLING_ENVS // 10
