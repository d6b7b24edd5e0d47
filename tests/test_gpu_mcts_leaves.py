"""GPU tests of the leaf-parallel search (several leaves per tree per round under virtual loss, include/ccx.h
ccx_mcts_*_leaves): bit for bit against the C oracle's restatement, the one-leaf calls unchanged, the fused net loop equal to
the round trips, and the callers (self-play, arena, drop-in MCTS) running with it."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle as orc
from conftest import GOLDEN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "leaves_oracle"))
import leaves_oracle as lvo  # noqa: E402

pytestmark = pytest.mark.gpu

WEIGHTS = os.path.join(GOLDEN, "good_model_weights.npz")


@pytest.fixture(scope="module")
def eng():
    from chinesecheckersagent_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def model():
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    return ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)


def dev(a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint64:
        a = a.view(np.int64)
    return torch.from_numpy(a).cuda()


def cfg4_roots(n, seed=0x5EED2026):
    st, _, _ = orc.step_random(orc.start_states(n), seed, 0, 6, nthreads=8)      # start advanced by 6 random plies
    return st


def oracle_evaluator(evaluator):
    """the oracle's test evaluator on the host, as a search_with callback"""
    def evaluate(leaf):
        st = np.zeros((8, leaf.shape[1]), dtype=np.uint64)
        st[:5] = leaf.cpu().numpy().view(np.uint64)
        p, v = lvo.eval_batch(orc.encode(st), evaluator)
        return dev(p), dev(v)
    return evaluate


def same_search(a, b):
    return (torch.equal(a["visits"], b["visits"]) and torch.equal(a["q"].view(torch.int64), b["q"].view(torch.int64))
            and torch.equal(a["pi"].view(torch.int64), b["pi"].view(torch.int64)) and torch.equal(a["n_nodes"], b["n_nodes"]))


@pytest.mark.parametrize("leaves", [2, 4, 8, 16])
@pytest.mark.parametrize("evaluator", [orc.EVAL_UNIFORM, orc.EVAL_HASH])
@pytest.mark.parametrize("pre_expand", [0, 1])
@pytest.mark.parametrize("ties", [None, (0xC0FFEE, 1000)])
def test_search_with_matches_the_oracle(eng, leaves, evaluator, pre_expand, ties):
    """visits, root Q (float64 bits), pi and node counts equal the leaf-parallel oracle (tests/leaves_oracle) on 128 cfg-4 roots"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    roots = cfg4_roots(128, seed=0x5EED2026 + leaves)
    n, num_itr, cpuct = roots.shape[1], 80, 1.5
    noise = np.random.default_rng(leaves).dirichlet(np.ones(128) * 0.3, size=n) if pre_expand else None
    kw = dict(random_ties=True, tie_seed=ties[0], tie_uid0=ties[1]) if ties else {}
    m = BatchedMCTS(eng, cpuct=cpuct, num_itr=num_itr, leaves_per_round=leaves, **kw)
    out = m.search_with(dev(roots), oracle_evaluator(evaluator), pre_expand=bool(pre_expand),
                        root_noise=dev(noise) if pre_expand else None)
    v, pi, q, nodes = lvo.mcts(roots, num_itr, cpuct, 1.0, pre_expand, evaluator, noise, nthreads=8, ties=ties, leaves=leaves)
    assert np.array_equal(out["visits"].cpu().numpy().astype(np.uint32), v)
    assert np.array_equal(out["q"].cpu().numpy().view(np.uint64), q.view(np.uint64))
    assert np.array_equal(out["pi"].cpu().numpy(), pi)
    assert np.array_equal(out["n_nodes"].cpu().numpy(), nodes)


def test_one_leaf_calls_equal_the_existing_calls(model):
    """the *_leaves entry points with leaves = 1 are the one-leaf search bit for bit"""
    from chinesecheckersagent_b200.engine import BatchedMCTS, _p
    e = model.eng
    roots = dev(cfg4_roots(96, seed=5))
    n = roots.shape[1]
    m = BatchedMCTS(e, num_itr=24)
    want = m.search_with(roots, model.evaluate_states)
    leaf = e.empty((5, n), torch.int64)
    e.call("ccx_mcts_set_tiebreak", 0, 0, 0)
    e.call("ccx_mcts_begin", n, _p(roots), 25, 0, -1, -1)
    e.call("ccx_mcts_leaf_budget", n, 1, 24)
    for _ in range(24):
        e.call("ccx_mcts_select_leaves", n, 1, 3.5, _p(leaf))
        p, v = model.evaluate_states(leaf)
        e.call("ccx_mcts_expand_backup_leaves", n, 1, _p(p), _p(v), None, 0, 0)
    got = m._outputs(n)
    e.call("ccx_mcts_finalize", n, 1.0, *[_p(t) for t in got])
    assert torch.equal(want["visits"], got[0]) and torch.equal(want["q"].view(torch.int64), got[2].view(torch.int64))
    want = m.search_net(roots)
    e.call("ccx_mcts_begin", n, _p(roots), 25, 0, -1, -1)
    e.call("ccx_mcts_run_net_leaves", n, 24, 1, 3.5, None, 0, 0)
    got = m._outputs(n)
    e.call("ccx_mcts_finalize", n, 1.0, *[_p(t) for t in got])
    assert torch.equal(want["visits"], got[0]) and torch.equal(want["q"].view(torch.int64), got[2].view(torch.int64))


def test_leaves_out_of_range_are_rejected(eng):
    from chinesecheckersagent_b200 import _lib
    from chinesecheckersagent_b200.engine import BatchedMCTS
    with pytest.raises(ValueError):
        BatchedMCTS(eng, leaves_per_round=17)
    BatchedMCTS(eng, num_itr=4).search(dev(cfg4_roots(2)))
    for bad in (0, 17):
        assert eng.L.ccx_mcts_select_leaves(eng.h, 2, bad, 3.5, None) == -1
        with pytest.raises(_lib.CcxError):
            eng.call("ccx_mcts_run_net_leaves", 2, 4, bad, 3.5, None, 0, 0)


@pytest.mark.parametrize("kernel", ["tc", "tc_acc"])
@pytest.mark.parametrize("leaves", [4, 8])
def test_fused_net_loop_equals_round_trips(model, kernel, leaves):
    """search_net (ccx_mcts_run_net_leaves) = search_with(model.evaluate_states) bit for bit; the direct, captured and
    replayed round graphs give the same trees; the batch is large enough (n * L positions) for the two-stream split, which
    must not change anything either"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    model.set_kernel(kernel)
    L, h = model.eng.L, model.eng.h
    try:
        for n, pre_expand in ((200, False), ((16400 if kernel == "tc_acc" else 8200) // leaves + 131, True)):
            st, _, _ = orc.step_random(orc.start_states(n), 21 + n, 0, 7, nthreads=8)
            roots = dev(st)
            noise = torch.rand((n, 128), dtype=torch.float64, device="cuda") if pre_expand else None
            m = BatchedMCTS(model.eng, num_itr=64, leaves_per_round=leaves)
            want = m.search_with(roots, model.evaluate_states, pre_expand=pre_expand, root_noise=noise)
            assert np.all(want["visits"].sum(1).cpu().numpy() == (64 if pre_expand else 63))
            before = L.ccx_graph_replays(h)
            for _ in range(3):                                           # direct, captured + launched, replayed
                got = m.search_net(roots, pre_expand=pre_expand, root_noise=noise)
                assert same_search(want, got)
            if not os.environ.get("CCX_NO_GRAPH"):
                assert L.ccx_graph_replays(h) - before == 2
            one = BatchedMCTS(model.eng, num_itr=64).search_net(roots, pre_expand=pre_expand, root_noise=noise)
            assert not torch.equal(one["visits"], want["visits"])         # not a no-op
    finally:
        model.set_kernel("tc")


def test_search_a_b_a_gives_the_same_a_and_overflow_is_reported(model):
    """no virtual loss or leaf record survives a search: A, B, A on one handle gives A twice, also when B overflowed its
    edge pool (n_nodes -1) and when B was a one-leaf search; a too small edge pool reports -1 with L > 1"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    a_roots, b_roots = dev(cfg4_roots(64, seed=1)), dev(cfg4_roots(64, seed=2))
    m = BatchedMCTS(model.eng, num_itr=40, leaves_per_round=8, random_ties=True, tie_seed=3)
    a1 = m.search_net(a_roots)
    small = BatchedMCTS(model.eng, num_itr=40, leaves_per_round=8, edges_per_tree=200).search_net(b_roots)
    assert np.all(small["n_nodes"].cpu().numpy() == -1)
    a2 = m.search_net(a_roots)
    assert same_search(a1, a2)
    m.search_net(b_roots)
    BatchedMCTS(model.eng, num_itr=40).search_net(b_roots)
    a3 = m.search_net(a_roots)
    assert same_search(a1, a3)
    tight = BatchedMCTS(model.eng, num_itr=40, leaves_per_round=8, edges_per_tree=200)
    res = tight.search_with(b_roots, model.evaluate_states)
    assert np.all(res["n_nodes"].cpu().numpy() == -1)
    assert same_search(a1, m.search_net(a_roots))
    assert model.eng.L.ccx_mcts_pool_bytes(model.eng.h) > 0


def test_selfplay_with_leaves_is_deterministic_and_well_formed(model):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay

    def run(compact, seed=9):
        sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=320, seed=seed, num_itr=16, max_iters=400, leaves_per_round=8)
        st = sp.play_games(360, compact=compact, compact_min=24)
        t = sp.collect()
        key = np.vstack([t["state"].cpu().numpy(), t["v_y"].cpu().numpy()[None].astype(np.int64),
                         (t["pi_y"].double() * torch.arange(1, 295, device=t["pi_y"].device)).sum(1).mul(1e6).round().long().cpu().numpy()[None]])
        order = np.lexsort(key)
        return st, t["board_x"].cpu().numpy()[order], t["pi_y"].cpu().numpy()[order], t["v_y"].cpu().numpy()[order], t
    a, b, c = run(False), run(False), run(True)
    assert a[0]["records"] > 0 and a[0]["games"] > 0
    for k in ("plies", "p1_wins", "p2_wins", "records", "games", "iterations"):
        assert a[0][k] == b[0][k] == c[0][k], k
    for i in (1, 2, 3):
        assert np.array_equal(a[i], b[i]) and np.array_equal(a[i], c[i])
    assert c[0]["compactions"] >= 1
    # the record format of the one-leaf self-play: root planes, pi on legal moves summing to 1, rewards +-1
    t = a[4]
    state = t["state"].cpu().numpy().view(np.uint64)
    full = np.zeros((8, state.shape[1]), dtype=np.uint64)
    full[:5] = state
    assert np.array_equal(t["board_x"].cpu().numpy(), orc.encode(full))
    pi = t["pi_y"].cpu().numpy()
    assert np.allclose(pi.sum(1), 1.0, atol=1e-5) and set(np.unique(t["v_y"].cpu().numpy())) <= {-1, 1}
    masks = orc.movegen(full)
    for i in range(0, pi.shape[0], max(1, pi.shape[0] // 100)):
        for act in np.nonzero(pi[i])[0]:
            cid, off = divmod(int(act), 49)
            assert (int(masks[cid, i]) >> ((off // 7) * 8 + off % 7)) & 1


def test_arena_pits_leaves_against_one_leaf(model):
    from chinesecheckersagent_b200.arena import BatchedArena
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)
    res = BatchedArena(model, other, 16, seed=3, num_itr=24, leaves_per_round=(8, 1)).play(max_plies=300)
    assert res["games"] == 16 and res["p1_wins"] + res["p2_wins"] > 0 and res["overflowed"] == 0
    again = BatchedArena(model, other, 16, seed=3, num_itr=24, leaves_per_round=(8, 1)).play(max_plies=300)
    assert res == again


def test_dropin_mcts_with_leaves_runs_the_reference_callers(model):
    """MCTS.LEAVES_PER_ROUND = 8: selfplay() (root expansion, Dirichlet noise, search) and an AiPlayer decision run through
    the unmodified callers; the root's visits add up to the simulations made"""
    import random

    from chinesecheckersagent_b200.board import Board
    from chinesecheckersagent_b200.MCTS import MCTS, Node
    from chinesecheckersagent_b200.player import AiPlayer
    from chinesecheckersagent_b200.selfplay import selfplay
    old = MCTS.LEAVES_PER_ROUND
    MCTS.LEAVES_PER_ROUND = 8
    try:
        np.random.seed(3); random.seed(3)
        hist, reward = selfplay(model, num_itr=24)
        assert (hist is None and reward is None) or (reward in (1, -1) and len(hist) > 0)
        tree = MCTS(Node(Board(engine=model.eng), 1), model, num_itr=40)
        pi, edge = tree.search()
        assert sum(e.stats['N'] for e in tree.root.edges) == 39 and abs(pi.sum() - 1) < 1e-12
        frm, to = AiPlayer(player_num=1, model=model, tree_tau=0.01).decide_move(Board(engine=model.eng))
        assert to in Board(engine=model.eng).get_valid_moves(1)[frm]

        class Foreign:                                   # not the package's net: predict() once per leaf slot
            calls = 0

            def predict(self, x):
                Foreign.calls += 1
                assert x.shape == (7, 7, 7)
                return np.full(294, 1 / 294.), 0.0
        tree = MCTS(Node(Board(engine=model.eng), 1), Foreign(), num_itr=33)
        tree.search()
        assert sum(e.stats['N'] for e in tree.root.edges) == 32
        assert Foreign.calls == 8 * (1 + 4)               # rounds: the root, then 8 + 8 + 8 + 8 selections
    finally:
        MCTS.LEAVES_PER_ROUND = old
