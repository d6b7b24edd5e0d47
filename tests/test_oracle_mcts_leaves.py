"""CPU oracle of the leaf-parallel search (several selections per tree per round under virtual loss): with one leaf per
round it is the one-leaf oracle bit for bit; with more it keeps the selection count, the node bound and leaves no
virtual loss behind, and it does change the search."""
import os
import sys

import numpy as np
import pytest

import oracle as orc
from conftest import GOLDEN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "leaves_oracle"))
import leaves_oracle as lvo  # noqa: E402

NUM_ITR = 60


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(GOLDEN, "mcts_golden.npz")))


def cfg4_roots(n, seed=0x5EED2026):
    st, _, _ = orc.step_random(orc.start_states(n), seed, 0, 6, nthreads=8)      # start advanced by 6 random plies
    return st


@pytest.mark.parametrize("evaluator", [orc.EVAL_UNIFORM, orc.EVAL_HASH])
@pytest.mark.parametrize("ties", [None, (0x1234, 7)])
@pytest.mark.parametrize("pre_expand", [0, 1])
def test_one_leaf_equals_the_one_leaf_oracle(gold, evaluator, ties, pre_expand):
    noise = gold["noise"] if pre_expand else None
    a = orc.mcts(gold["roots"], NUM_ITR, 3.5, 1.0, pre_expand, evaluator, noise, nthreads=8, ties=ties)
    stats = {}
    b = lvo.mcts(gold["roots"], NUM_ITR, 3.5, 1.0, pre_expand, evaluator, noise, nthreads=8, ties=ties, leaves=1, stats=stats)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))        # root Q, float64 bits
    assert not stats["vl_left"].any()


@pytest.mark.parametrize("leaves", [2, 8])
@pytest.mark.parametrize("evaluator", [orc.EVAL_UNIFORM, orc.EVAL_HASH])
@pytest.mark.parametrize("ties", [None, (0x1234, 7)])
@pytest.mark.parametrize("pre_expand", [0, 1])
def test_several_leaves_keep_the_search_invariants(gold, leaves, evaluator, ties, pre_expand):
    roots = np.concatenate([gold["roots"], cfg4_roots(32)], axis=1)
    noise = np.tile(gold["noise"][:1], (roots.shape[1], 1)) if pre_expand else None
    # cpuct 1: Q weighs enough against U that virtual losses steer the descents (at 3.5 and 60 simulations the hash
    # evaluator's trees are so wide that most rounds pick the same edges either way)
    one = orc.mcts(roots, NUM_ITR, 1.0, 1.0, pre_expand, evaluator, noise, nthreads=8, ties=ties)
    stats = {}
    v, pi, q, nodes = lvo.mcts(roots, NUM_ITR, 1.0, 1.0, pre_expand, evaluator, noise, nthreads=8, ties=ties, leaves=leaves,
                               stats=stats)
    live = one[0].sum(1) > 0                                  # roots that are not already won
    assert np.array_equal(v.sum(1)[live], one[0].sum(1)[live])
    assert np.all(v.sum(1)[live] == (NUM_ITR if pre_expand else NUM_ITR - 1))
    assert np.all(stats["visited"] <= NUM_ITR + 2)
    assert np.all(stats["visited"] >= 2)
    assert not stats["vl_left"].any()
    assert np.allclose(pi.sum(1)[live], 1.0)
    if evaluator == orc.EVAL_HASH:                             # (with uniform priors and v = 0 the visits spread the same way)
        assert (v != one[0]).any(axis=1).sum() >= 4            # not a no-op


def test_terminal_leaves_and_duplicates_occur():
    """Late positions (a greedy game played close to its end) reach wins inside the horizon: terminal selections and
    duplicate selections both happen within rounds, and the invariants still hold."""
    st = orc.play_greedy(orc.start_states(16), 0xABC, max_plies=36)
    stats = {}
    v, pi, q, nodes = lvo.mcts(st, NUM_ITR, 1.0, 1.0, 1, orc.EVAL_HASH, None, nthreads=8, leaves=16, stats=stats)
    live = v.sum(1) > 0
    assert live.sum() >= 8
    assert np.all(v.sum(1)[live] == NUM_ITR)
    assert np.any(stats["visited"][live] < NUM_ITR + 1)        # some selections were duplicates or repeated terminals
    assert not stats["vl_left"].any()


def test_eval_batch_is_the_search_evaluator():
    st = cfg4_roots(8)
    planes = orc.encode(st)
    p, v = lvo.eval_batch(planes, orc.EVAL_HASH)
    assert p.shape == (8, 294) and v.shape == (8,)
    assert np.all((p >= 0) & (p < 1)) and np.all((v >= -1) & (v < 1))
    p2, v2 = lvo.eval_batch(planes, orc.EVAL_HASH)
    assert np.array_equal(p, p2) and np.array_equal(v, v2)
    pu, vu = lvo.eval_batch(planes, orc.EVAL_UNIFORM)
    assert np.all(pu == 1 / 294.) and not vu.any()
