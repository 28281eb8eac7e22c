"""CPU: the softmax exploration rule of rlrm_set_exploration as the CPU oracle restates it (tests/softmax_oracle.c).

* rlrm_exp against math.exp on about 10^6 points (dense near 0, uniform over [-745, 0], the cutoff and the subnormal edge,
  consecutive doubles across every range-reduction boundary): within 2 ULP, exp(0) == 1, monotone, +0 below the cutoff;
* selection frequencies over 2^20 consecutive Philox words against numpy's softmax probabilities (chi-square with a fixed
  seed, so the outcome is deterministic), on ties, a -3000 entry, n_actions 1-3 and a temperature so small that only the
  maxima survive;
* the oracle's select path (SoftmaxOracle) picks #{j : w1 >= T_j}."""
import math

import numpy as np
import pytest
from scipy import stats

import multiagent_rlrm_b200 as P
import oracle as O
import softmax_oracle as SO
import philox

LN2 = math.log(2.0)
CUTOFF = float.fromhex("-0x1.74910d52d3052p+9")  # below: rlrm_exp returns +0


def _ulps(a, b):
    """distance in units in the last place of non-negative doubles (their bit patterns are ordered like their values)"""
    return np.abs(a.view(np.int64) - b.view(np.int64))


def _points():
    rng = np.random.default_rng(2024)
    dense = -np.abs(rng.standard_normal(200_000)) * 10.0 ** rng.integers(-300, 1, 200_000)
    uniform = -rng.uniform(0.0, 745.0, 500_000)
    tiny = -rng.uniform(0.0, 1.0, 100_000)
    sub = -rng.uniform(700.0, 746.0, 100_000)  # the subnormal range starts at ln(2^-1022) = -708.4
    edges = [0.0, -0.0, -5e-324, -1e-300, CUTOFF, np.nextafter(CUTOFF, 0.0), np.nextafter(CUTOFF, -np.inf), -745.0, -746.0,
             -708.3964185322641, -708.4, -709.0, -1022 * LN2, -1074 * LN2, -1075 * LN2]
    # 64 consecutive doubles on each side of every boundary where rint(x * log2e) changes k
    walk = []
    for k in range(0, 1076):
        bits = np.float64(-(k + 0.5) * LN2).view(np.int64)
        walk.append((bits + np.arange(-64, 64, dtype=np.int64)).view(np.float64))  # negative doubles: +1 in the bits is one step down
    x = np.concatenate([dense, uniform, tiny, sub, np.array(edges, dtype=np.float64)] + walk)
    return np.minimum(x, 0.0)


def test_exp_within_two_ulp_of_math_exp():
    x = _points()
    assert x.size > 1_000_000
    got = SO.exp(x)
    ref = np.array([math.exp(v) for v in x])
    u = _ulps(got, ref)
    worst = int(np.argmax(u))
    assert u.max() <= 2, f"rlrm_exp({x[worst]!r}) = {got[worst]!r}, math.exp = {ref[worst]!r}: {u.max()} ULP"
    # mostly correctly rounded: a coarse guard against a constant typo that stays under 2 ULP
    assert np.mean(u == 0) > 0.9


def test_exp_edges():
    assert SO.exp(np.array([0.0, -0.0])).tolist() == [1.0, 1.0]
    below = np.array([np.nextafter(CUTOFF, -np.inf), -746.0, -1e4, -np.inf, -1e308])
    assert np.all(SO.exp(below) == 0.0) and not np.any(np.signbit(SO.exp(below)))
    # the cutoff is the double nearest ln(2^-1075): from the next double up exp(x) rounds to the smallest subnormal
    edge = np.array([CUTOFF, np.nextafter(CUTOFF, 0.0)])
    assert SO.exp(edge).tolist() == [math.exp(v) for v in edge] == [0.0, 5e-324]
    assert SO.exp(np.array([-1.0]))[0] == math.exp(-1.0)


def test_exp_monotone():
    x = np.sort(_points())
    y = SO.exp(x)
    bad = np.nonzero(np.diff(y) < 0)[0]
    assert bad.size == 0, f"rlrm_exp decreases between {x[bad[0]]!r} and {x[bad[0] + 1]!r}"


# ----------------------------------------------------------------------------------------------------------------------
# selection frequencies
# ----------------------------------------------------------------------------------------------------------------------
N_WORDS = 1 << 20


def _w1_words():
    """w1 of 2^20 consecutive Philox counters (iterations 0 .. 2^20 - 1 of instance 0, agent 0) under a fixed key"""
    t = np.arange(N_WORDS, dtype=np.uint64)
    _w0, w1, _w2, _w3 = philox.philox4x32_10(t, 0, 0, 0, 0x1234567, 0x89ABCDE)
    return w1.astype(np.uint64)


def _numpy_softmax(row, tau):
    z = np.asarray(row, dtype=np.float64) / tau
    z = z - z.max()
    p = np.exp(z)
    return p / p.sum()


ROWS = [  # (row, temperature)
    ([1.0, 2.0, 3.0, 4.0], 1.0),
    ([0.5, 0.5, 0.5, 0.5], 0.3),  # ties: uniform
    ([2.0, 2.0, -1.0, 0.0], 0.7),  # tied maxima
    ([0.0, -3000.0, 1.0, 0.25], 1.0),  # one entry underflows: never chosen
    ([-3000.0, 0.0, 0.0, 0.1], 2.5),
    ([0.1, 0.2], 0.05),  # n_actions = 2
    ([3.0, -1.0, 0.0], 10.0),  # n_actions = 3
    ([7.0], 1.0),  # n_actions = 1
    ([1.0, 1.0, 0.9999, 1.0], 1e-9),  # only the maxima survive: uniform among them
    ([-2.0, 5.0, 5.0, 4.99], 1e-12),
    ([1e-3, -1e-3, 0.0, 2e-3], 1e-3),
]


@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("row,tau", ROWS)
def test_selection_frequencies_match_numpy_softmax(row, tau, real):
    w1 = _w1_words()
    thr = SO.softmax_thresholds(row, tau, real)
    assert thr.size == len(row) - 1 and np.all(np.diff(thr.astype(np.int64)) >= 0) and np.all(thr <= 1 << 32)
    actions = np.searchsorted(thr, w1, side="right")  # #{j : w1 >= T_j}
    counts = np.bincount(actions, minlength=len(row))
    dt = np.float32 if real == "f32" else np.float64
    p = _numpy_softmax(np.asarray(row, dtype=dt).astype(np.float64), tau)
    zero = p < 1e-300
    assert np.all(counts[zero] == 0), (row, tau, counts)
    live = ~zero
    if live.sum() == 1:
        assert counts[live][0] == N_WORDS
        return
    exp_counts = p[live] / p[live].sum() * N_WORDS
    chi2 = stats.chisquare(counts[live], exp_counts)
    assert chi2.pvalue > 1e-4, (row, tau, counts, exp_counts)


def test_small_temperature_is_uniform_among_maxima():
    for row in ([1.0, 1.0, 0.9999, 1.0], [-2.0, 5.0, 5.0, 4.99]):
        thr = SO.softmax_thresholds(row, 1e-9, "f64")
        m = max(row)
        w = np.array([1.0 if v == m else 0.0 for v in row])  # exact weights: maxima 1, the rest underflow to +0
        c = np.cumsum(w)
        assert thr.tolist() == [int(np.ceil(cj / c[-1] * 2.0 ** 32)) for cj in c[:-1]]


def test_equal_rows_split_the_words_evenly():
    thr = SO.softmax_thresholds([0.25, 0.25, 0.25, 0.25], 1.0, "f32")
    assert thr.tolist() == [1 << 30, 2 << 30, 3 << 30]
    thr = SO.softmax_thresholds([0.0, 0.0, 0.0], 0.5, "f64")
    assert thr.tolist() == [int(np.ceil(1 / 3 * 2.0 ** 32)), int(np.ceil(2 / 3 * 2.0 ** 32))]


# ----------------------------------------------------------------------------------------------------------------------
# the oracle's select path
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("n_actions", [1, 2, 3, 4])
def test_oracle_select_uses_the_thresholds(real, n_actions):
    sc = P.Scenario(env="frozen_lake", map_name="map1", starts=[(0, 0), (3, 3)], rm_transitions=[("u0", (1, 1), "u1", 1.0)],
                    detector_positions=[(1, 1)], algo="ql", seed=7, table_dtype=real)
    c = P.compile_scenario(sc)
    c.config.n_actions = n_actions
    n, tau = 40, 0.37
    o = SO.SoftmaxOracle(c, n, tau)
    greedy = O.Oracle(c, n)
    rng = np.random.default_rng(n_actions)
    for ora in (o, greedy):
        ora.reset()
    q = rng.choice([0.0, 1.0, -0.5, 0.3, -3000.0], size=o.q.shape).astype(o.q.dtype)
    o.q[...] = q
    greedy.q[...] = q
    draws = rng.integers(0, 1 << 32, size=(n, 2, 4), dtype=np.uint64).astype(np.uint32)
    got = o.select_action(draws=draws)
    slots = o.unpack()
    for i in range(n):
        for a in range(2):
            row = o.q[i * 2 + a, slots["cell"][i, a] * c.config.n_rm_states + slots["q"][i, a]][:n_actions]
            thr = SO.softmax_thresholds(row, tau, real)
            assert got[i, a] == int(np.sum(np.uint64(draws[i, a, 1]) >= thr))
    # greedy evaluation is unchanged, and the epsilon-greedy oracle is unaffected by the softmax one
    assert np.array_equal(o.select_action(draws=draws, best=True), greedy.select_action(draws=draws, best=True))
    o2 = O.Oracle(c, n)
    o2.reset()
    o2.q[...] = q
    assert np.array_equal(o2.select_action(draws=draws), greedy.select_action(draws=draws))
