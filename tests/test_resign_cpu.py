"""CPU: the self-play resignation rule of include/ccx.h as the host restates it (tests/resign_ref.py) — the resign value in the
kernels' summation order, the streak, the windowed minimum — and the threshold calibration of selfplay.suggest_resign_threshold."""
import math

import numpy as np
import pytest

import resign_ref


def lane_order_sum(x):
    """the warp order with NumPy: per-lane sums over four chunks, then the butterfly"""
    a = np.zeros(128)
    a[:len(x)] = x
    lanes = a.reshape(4, 32)
    s = ((lanes[0] + lanes[1]) + lanes[2]) + lanes[3]
    for off in (16, 8, 4, 2, 1):
        s = s + s[np.arange(32) ^ off]
    return s[0]


def test_value_of_hand_built_roots():
    # ties for the maximal N: the first such edge's Q
    N, Q = [3, 5, 5, 1], [0.5, -0.25, 0.75, 1.0]
    v = (3 * 0.5 + 5 * -0.25 + 5 * 0.75 + 1.0) / 14
    assert resign_ref.resign_value(N, Q) == max(v, -0.25)
    # the root value wins when the best child is worse
    N, Q = [2, 9, 1], [0.9, -0.5, 1.0]
    assert resign_ref.resign_value(N, Q) == (2 * 0.9 - 4.5 + 1.0) / 12
    # zero visits: no value
    assert math.isnan(resign_ref.resign_value([0, 0, 0], [0.0, 0.0, 0.0]))
    assert math.isnan(resign_ref.resign_value([], []))
    # a single edge: both terms are its Q
    assert resign_ref.resign_value([7], [-0.375]) == -0.375
    # unvisited edges add nothing
    assert resign_ref.resign_value([0, 4, 0], [0.0, 0.25, 0.0]) == 0.25


def test_value_of_126_edges_follows_the_warp_order():
    rng = np.random.default_rng(3)
    for _ in range(50):
        N = rng.integers(0, 40, 126).astype(np.uint32)
        W = rng.uniform(-1, 1, 126) * N
        Q = np.where(N > 0, W / np.maximum(N, 1), 0.0)
        r = resign_ref.resign_value(list(N), list(Q))
        v = lane_order_sum(N.astype(np.float64) * Q) / lane_order_sum(N.astype(np.float64))
        assert r == max(v, Q[int(np.argmax(N))])
        assert abs(v - math.fsum(N * Q) / math.fsum(N)) < 1e-12


@pytest.mark.parametrize("plies", range(1, 9))
def test_streak_rule(plies):
    rng = np.random.default_rng(plies)
    t = 0.0
    for _ in range(200):
        k = int(rng.integers(1, 60))
        vals = [(i & 1, float(x)) for i, x in enumerate(rng.uniform(-0.3, 0.6, k))]
        at, would, _ = resign_ref.track_game(vals, t, plies, probe=False)
        expect = None                                   # first ply whose player's last `plies` values are all below t
        for i, (p, _) in enumerate(vals):
            mine = [r for q, r in vals[:i + 1] if q == p]
            if len(mine) >= plies and all(r < t for r in mine[-plies:]):
                expect = i
                break
        assert at == expect and would == (None if expect is None else vals[expect][0])
        pat, pwould, _ = resign_ref.track_game(vals, t, plies, probe=True)
        assert pat is None and pwould == would
    # a ply at or above the threshold resets the streak
    assert resign_ref.track_game([(0, -0.5), (0, 0.0), (0, -0.5)], 0.0, 2, False)[0] is None
    assert resign_ref.track_game([(0, -0.5), (0, -0.5)], 0.0, 2, False)[0] == 1
    # threshold -1 never resigns (r >= -1)
    assert resign_ref.track_game([(0, -1.0)] * 20, -1.0, 1, False)[:2] == (None, None)


@pytest.mark.parametrize("plies", [1, 2, 3, 8])
def test_windowed_minimum(plies):
    rng = np.random.default_rng(10 + plies)
    for _ in range(100):
        vals = [(i & 1, float(x)) for i, x in enumerate(rng.uniform(-1, 1, int(rng.integers(1, 40))))]
        _, _, wmin = resign_ref.track_game(vals, -1.0, plies, probe=True)
        for p in (0, 1):
            mine = [r for q, r in vals if q == p]
            expect = min((max(mine[i - plies + 1:i + 1]) for i in range(plies - 1, len(mine))), default=math.inf)
            assert wmin[p] == expect
            # the window minimum is the largest threshold at which the player never resigns
            if expect < math.inf:
                assert resign_ref.track_game([(0, r) for r in mine], expect, plies, False)[0] is None
                assert resign_ref.track_game([(0, r) for r in mine], np.nextafter(expect, 2), plies, False)[0] is not None


def test_threshold_suggestion():
    from chinesecheckersagent_b200.selfplay import suggest_resign_threshold as sugg
    assert sugg([], 0.05) == -1.0
    assert sugg(np.full(40, 0.2), 0.05) == 0.2                  # rate at 0.2 is 0, just above it 1
    assert sugg([0.3], 0.0) == 0.3 and sugg([0.3], 1.0) == 1.0
    assert sugg([-0.5, math.inf], 0.5) == 1.0                     # clipped to 1
    with pytest.raises(ValueError):
        sugg([0.1], 1.5)
    rng = np.random.default_rng(7)
    for m in (1, 2, 19, 100, 1000):
        s = rng.uniform(-1, 0.8, m)
        s[rng.integers(0, m, m // 4)] = s[0]                      # ties
        for fp in (0.0, 0.01, 0.02, 0.05, 0.1, 0.5):
            t = sugg(s, fp)
            rate = lambda x: np.count_nonzero(s < x) / m       # noqa: E731
            assert rate(t) <= fp
            assert t == 1.0 or rate(np.nextafter(t, 2)) > fp    # the largest such threshold
