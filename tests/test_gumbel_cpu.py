"""CPU checks of the Gumbel search's shared pieces and of its C restatement: the sequential-halving schedule equals mctx's
get_sequence_of_considered_visits, ccx_fpmath's log / exp are within 2 ulp of libm, and the restatement's results are well
formed (the improved policy is a distribution on the legal moves, the action is a considered move, m = 1 at scale 0 plays
the top-prior move)."""
import math
import os
import sys

import numpy as np
import pytest

import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "gumbel_oracle"))
import gumbel_oracle as gmo  # noqa: E402


def mctx_sequence(max_num_considered_actions, num_simulations):
    """mctx/_src/seq_halving.py, get_sequence_of_considered_visits (Apache-2.0), as published"""
    if max_num_considered_actions <= 1:
        return tuple(range(num_simulations))
    log2max = int(math.ceil(math.log2(max_num_considered_actions)))
    sequence = []
    visits = [0] * max_num_considered_actions
    num_considered = max_num_considered_actions
    while len(sequence) < num_simulations:
        num_extra_visits = max(1, int(num_simulations / (log2max * num_considered)))
        for _ in range(num_extra_visits):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, num_considered // 2)
    return tuple(sequence[:num_simulations])


def test_schedule_equals_mctx():
    for m in range(1, 33):
        for sims in range(1, 401):
            assert tuple(gmo.considered_visits(m, sims).tolist()) == mctx_sequence(m, sims), (m, sims)


def ulps(a, b):
    ia, ib = np.array([a, b]).view(np.int64)
    return abs(int(ia) - int(ib))


def test_fpmath_within_two_ulp_of_libm():
    rng = np.random.default_rng(7)
    xs = np.concatenate([np.exp(rng.uniform(-745, 709, 20000)), rng.uniform(0.5, 2.0, 20000), 1 + rng.uniform(-1e-6, 1e-6, 2000),
                         [5e-324, 2.2250738585072014e-308, 1e-300, 0.5, 1.0, 2.0, 1e300, 1.7976931348623157e308]])
    worst = max(ulps(gmo.fm_log(x), math.log(x)) for x in xs)
    assert worst <= 2, worst
    ys = np.concatenate([rng.uniform(-745, 709, 20000), rng.uniform(-1, 1, 20000), rng.uniform(-1e-8, 1e-8, 2000),
                         [0.0, -0.0, 1.0, -1.0, 709.78, -708.39, -744.0]])
    worst = max(ulps(gmo.fm_exp(y), math.exp(y)) for y in ys)
    assert worst <= 2, worst
    assert gmo.fm_exp(-746.0) == 0.0 and gmo.fm_exp(710.0) == math.inf and gmo.fm_log(1.0) == 0.0


def roots(n, seed):
    st, _, _ = orc.step_random(orc.start_states(n), seed, 0, 6, nthreads=8)
    return st


@pytest.mark.parametrize("evaluator", [gmo.EVAL_UNIFORM, gmo.EVAL_HASH])
@pytest.mark.parametrize("considered,sims", [(16, 32), (4, 64), (200, 16), (2, 5)])
def test_restatement_is_well_formed(evaluator, considered, sims):
    st = roots(48, 11 + sims)
    out = gmo.mcts(st, sims, pre_expand=1, evaluator=evaluator, considered=considered, seed=5, nthreads=8)
    masks = orc.movegen(st)
    for i in range(st.shape[1]):
        legal = np.zeros(294, dtype=bool)
        for a in range(294):
            cid, off = divmod(a, 49)
            legal[a] = (int(masks[cid, i]) >> ((off // 7) * 8 + off % 7)) & 1
        pi = out["pi"][i]
        assert abs(pi.sum() - 1.0) < 1e-12 and np.all(pi >= 0) and not np.any(pi[~legal] > 0)
        assert legal[out["action"][i]] and out["in_considered"][i] == 1
        assert out["visits"][i].sum() == sims                     # pre_expand: every simulation passes the root
        assert out["n_nodes"][i] >= 1 + legal.sum()               # root + one node per root edge, at least


def test_one_considered_move_at_scale_zero_plays_the_top_prior_move():
    st = roots(32, 3)
    out = gmo.mcts(st, 8, pre_expand=1, evaluator=gmo.EVAL_HASH, considered=1, scale=0.0, nthreads=8)
    full = np.zeros((8, st.shape[1]), dtype=np.uint64)
    full[:] = st
    p, _ = gmo.eval_batch(orc.encode(full), gmo.EVAL_HASH)
    masks = orc.movegen(st)
    for i in range(st.shape[1]):
        legal = [a for a in range(294) if (int(masks[a // 49, i]) >> (((a % 49) // 7) * 8 + (a % 49) % 7)) & 1]
        assert out["action"][i] == max(legal, key=lambda a: (p[i, a], -a))
        assert out["visits"][i][out["action"][i]] == 8            # the only considered move takes every simulation


def test_scale_and_seed_change_the_search():
    st = roots(32, 4)
    a = gmo.mcts(st, 24, evaluator=gmo.EVAL_HASH, seed=1, nthreads=8)
    b = gmo.mcts(st, 24, evaluator=gmo.EVAL_HASH, seed=2, nthreads=8)
    c = gmo.mcts(st, 24, evaluator=gmo.EVAL_HASH, seed=2, uids=np.arange(32), nthreads=8)
    assert not np.array_equal(a["visits"], b["visits"])
    assert all(np.array_equal(b[k], c[k]) for k in b)            # uid0 + i and explicit uids i are the same trees
