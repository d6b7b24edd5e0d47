"""CPU oracle of tree reuse (persistent trees re-rooted by state match, include/ccx.h ccx_mcts_begin_reuse): without a carried
tree every search is today's leaf-parallel oracle bit for bit; a carried tree holds the original subtree's statistics and
no virtual loss."""
import os
import sys

import numpy as np
import pytest

import oracle as orc

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "leaves_oracle"))
import leaves_oracle as lvo  # noqa: E402
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "reuse_oracle"))
import reuse_oracle as rvo  # noqa: E402

SIMS = 40


def cfg4_roots(n, seed=0x5EED2026):
    st, _, _ = orc.step_random(orc.start_states(n), seed, 0, 6, nthreads=8)      # start advanced by 6 random plies
    return st


def play(st, acts):
    """apply policy index acts[i] (checker id * 49 + destination r*7+c) to the side to move of every state"""
    acts = np.asarray(acts, dtype=np.int64)
    side = (st[4] >> np.uint64(48)) & np.uint64(1)
    cells = np.where(side == 1, st[3], st[2])
    cid, off = acts // 49, acts % 49
    frm = ((cells >> (np.uint64(8) * cid.astype(np.uint64))) & np.uint64(0xFF)).astype(np.uint8)
    to = ((off // 7) * 8 + off % 7).astype(np.uint8)
    return orc.apply(st, frm, to)[0]


def best(visits):
    return visits.argmax(1)


def most_visited_reply(f, i, act):
    """the reply with the most visits below tree i's move `act` (the highest prior when none has a visit yet)"""
    N, _, P = f.child_stats(i, act)
    return N.argmax() if N.any() else P.argmax()


@pytest.mark.parametrize("leaves", [1, 4])
@pytest.mark.parametrize("evaluator", [orc.EVAL_UNIFORM, orc.EVAL_HASH])
@pytest.mark.parametrize("ties", [None, (0x1234, 7)])
@pytest.mark.parametrize("pre_expand", [0, 1])
def test_no_carry_equals_the_leaves_oracle(leaves, evaluator, ties, pre_expand):
    """carry = 0 (every tree fresh) and roots without a match in the old trees: each search is lvo.mcts bit for bit"""
    st = cfg4_roots(48, seed=11 + leaves)
    noise = np.random.default_rng(3).dirichlet(np.ones(128) * 0.3, size=48) if pre_expand else None
    f = rvo.Forest()
    for ply, carry in enumerate((0, 0, 3)):
        if ply == 2:
            st = cfg4_roots(48, seed=99)                                         # unrelated roots: nothing matches
        reused = f.begin(st, SIMS + 1, carry, noise=noise if pre_expand else None)
        assert not reused.any()
        f.search(SIMS + pre_expand, leaves, 3.5, evaluator, noise=noise, ties=ties)
        stats = {}
        got = f.finalize(stats=stats)
        want = lvo.mcts(st, SIMS, 3.5, 1.0, pre_expand, evaluator, noise, nthreads=8, ties=ties, leaves=leaves)
        for x, y in zip(got, want):
            assert np.array_equal(x, y)
        assert np.array_equal(got[2].view(np.uint64), want[2].view(np.uint64))
        assert not stats["vl_left"].any()
        st = play(st, best(got[0]))


@pytest.mark.parametrize("leaves", [1, 4])
def test_carried_subtree_keeps_its_statistics(leaves):
    """depth 1 (one move) and depth 2 (two moves): the carried root's N, W, P are the original subtree's, no virtual loss is
    left, and the following search adds exactly its selections"""
    st = cfg4_roots(48, seed=5)
    f = rvo.Forest()
    f.begin(st, SIMS + 1, 3)
    f.search(SIMS, leaves, 3.5, orc.EVAL_HASH)
    v, _, _, _ = f.finalize()
    acts = best(v)
    want = [f.child_stats(i, a) for i, a in enumerate(acts)]
    st1 = play(st, acts)
    reused = f.begin(st1, SIMS + 1, 3)
    assert (reused == 1).sum() >= 40 and set(np.unique(reused)) <= {0, 1}
    stats = {}
    v1, _, _, _ = f.finalize(stats=stats)
    for i in np.nonzero(reused == 1)[0]:
        N, W, P = want[i]
        assert np.array_equal(v1[i], N) and np.array_equal(stats["W"][i], W) and np.array_equal(stats["P"][i], P)
    f.search(SIMS, leaves, 3.5, orc.EVAL_HASH)
    v2, _, _, _ = f.finalize(stats=stats)
    assert not stats["vl_left"].any()
    assert np.array_equal(v2.sum(1), v1.sum(1) + np.where(reused == 1, SIMS, SIMS - 1))
    # depth 2: the move of the search just made and the reply that the carried tree explored most
    a1 = best(v2)
    reply = np.array([most_visited_reply(f, i, a) for i, a in enumerate(a1)])
    st2 = play(play(st1, a1), reply)
    r2 = f.begin(st2, SIMS + 1, 3)
    assert (r2 == 2).sum() > 0 and set(np.unique(r2)) <= {0, 2}


def test_carry_limit_and_remap():
    """a small carry falls back to fresh trees; prev moves sources between trees, -1 and out-of-range entries start fresh"""
    st = cfg4_roots(32, seed=8)
    E = 20000                                     # one edge budget for every begin below: the pool is kept
    trees = []
    for _ in range(2):
        f = rvo.Forest()
        f.begin(st, 201, 1, edges_per_tree=E)
        f.search(200, 1, 3.5, orc.EVAL_HASH)
        trees.append(f)
    v, _, _, _ = f.finalize()
    st1 = play(st, best(v))
    big = trees[0].begin(st1, 201, 1, edges_per_tree=E)
    small = trees[1].begin(st1, 11, 1, edges_per_tree=E)      # carry 1 of a 10-simulation search: at most 12 visits
    assert (big == 1).all() and (small == 0).sum() > 16
    f = trees[0]
    f.search(SIMS, 1, 3.5, orc.EVAL_HASH)
    v, _, _, _ = f.finalize()
    st2 = play(st1, best(v))
    f.begin(st2, 201, 1, edges_per_tree=E)
    f.search(SIMS, 1, 3.5, orc.EVAL_HASH)
    v, _, _, _ = f.finalize()
    st3 = play(st2, best(v))
    perm = np.random.default_rng(1).permutation(32)
    prev = perm.copy()
    prev[:3] = (-1, 32, 1 << 40)
    keep = f.begin(st3, 201, 1, edges_per_tree=E)
    f.search(SIMS, 1, 3.5, orc.EVAL_HASH)
    v, _, _, _ = f.finalize()
    st4 = play(st3, best(v))
    reused = f.begin(st4[:, perm], 201, 1, prev=prev, edges_per_tree=E)
    assert keep.sum() > 16 and not reused[:3].any() and reused[3:].sum() > 10
    # inactive roots (status byte set, min_ply 0) stay inactive: node count -2, no visits
    st4 = st4[:, perm]
    f.search(SIMS, 1, 3.5, orc.EVAL_HASH)
    v, _, _, _ = f.finalize()
    st4 = play(st4, best(v))
    st4[4, :4] |= np.uint64(1 << 56)
    r = f.begin(st4, 201, 1, min_ply=0, edges_per_tree=E)
    assert np.array_equal(r[:4], [-2] * 4) and r[4:].sum() > 10
    f.search(SIMS, 1, 3.5, orc.EVAL_HASH)
    v, _, _, nodes = f.finalize()
    assert np.array_equal(nodes[:4], [-2] * 4) and not v[:4].any()
    f.invalidate()                                           # a new net: nothing is carried
    assert not f.begin(play(st4, best(v)), 201, 1, min_ply=0, edges_per_tree=E)[4:].any()
