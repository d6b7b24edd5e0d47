"""GPU tests of the Gumbel search (include/ccx.h ccx_mcts_set_gumbel): bit for bit against the C restatement
(tests/gumbel_oracle), the fused net loop equal to the round trips, the PUCT searches of the same engine unaffected, and
self-play and the arena running with it."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle as orc
from conftest import GOLDEN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "gumbel_oracle"))
import gumbel_oracle as gmo  # noqa: E402

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


def cfg4_roots(n, seed=0x5EED2026, plies=6):
    """start advanced by `plies` random plies; plies < 0: randomised positions (Board(randomised=True)) advanced by 2"""
    st = orc.random_states(n, seed) if plies < 0 else orc.start_states(n)
    st, _, _ = orc.step_random(st, seed, 0, max(plies, 2), nthreads=8)
    return st


def oracle_evaluator(evaluator):
    def evaluate(leaf):
        st = np.zeros((8, leaf.shape[1]), dtype=np.uint64)
        st[:5] = leaf.cpu().numpy().view(np.uint64)
        p, v = gmo.eval_batch(orc.encode(st), evaluator)
        return dev(p), dev(v)
    return evaluate


def check_equal(out, want):
    assert np.array_equal(out["visits"].cpu().numpy().astype(np.uint32), want["visits"])
    assert np.array_equal(out["q"].cpu().numpy().view(np.uint64), want["q"].view(np.uint64))
    assert np.array_equal(out["pi"].cpu().numpy().view(np.uint64), want["pi"].view(np.uint64))
    assert np.array_equal(out["action"].cpu().numpy(), want["action"])
    assert np.array_equal(out["n_nodes"].cpu().numpy(), want["n_nodes"])


CASES = [  # (plies of the roots, pre_expand, considered, simulations, scale, evaluator)
    (6, 0, 16, 175, 1.0, gmo.EVAL_HASH), (6, 1, 16, 175, 1.0, gmo.EVAL_UNIFORM), (6, 1, 1, 16, 0.0, gmo.EVAL_HASH),
    (6, 0, 2, 16, 1.0, gmo.EVAL_HASH), (6, 1, 4, 2, 1.0, gmo.EVAL_HASH), (40, 1, 200, 16, 1.0, gmo.EVAL_HASH),
    (40, 0, 4, 1, 1.0, gmo.EVAL_UNIFORM), (40, 1, 16, 1, 0.0, gmo.EVAL_HASH), (80, 1, 200, 175, 0.0, gmo.EVAL_UNIFORM),
    (-1, 0, 16, 175, 1.0, gmo.EVAL_HASH), (-1, 1, 2, 16, 0.0, gmo.EVAL_HASH),
]


@pytest.mark.parametrize("plies,pre_expand,considered,sims,scale,evaluator", CASES)
def test_search_with_matches_the_oracle(eng, plies, pre_expand, considered, sims, scale, evaluator):
    """visits, root Q and improved pi (float64 bits), action and node counts equal the restatement on 96 roots (cfg-4 roots
    after 6 random plies, mid-game roots after 40 or 80, randomised positions)"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    roots = cfg4_roots(96, seed=(plies + 2) * 1000 + sims, plies=plies)
    m = BatchedMCTS(eng, num_itr=sims, gumbel=True, gumbel_considered=considered, gumbel_scale=scale, gumbel_seed=0xBEEF,
                    tie_uid0=500)
    out = m.search_with(dev(roots), oracle_evaluator(evaluator), pre_expand=bool(pre_expand))
    want = gmo.mcts(roots, sims, pre_expand, evaluator, considered=considered, scale=scale, seed=0xBEEF, uid0=500, nthreads=8)
    check_equal(out, want)


def test_slot_ids_key_the_draws(eng):
    """with slot ids set, tree i draws as uid slot_ids[i]: a permuted batch gives the permuted results"""
    from chinesecheckersagent_b200.engine import BatchedMCTS, _p
    roots = cfg4_roots(64, seed=77)
    uids = np.arange(1000, 1064)[::-1].copy()
    ids = dev(uids)
    eng.call("ccx_set_slot_ids", _p(ids))
    try:
        out = BatchedMCTS(eng, num_itr=32, gumbel=True, gumbel_seed=9).search_with(dev(roots), oracle_evaluator(gmo.EVAL_HASH))
    finally:
        eng.call("ccx_set_slot_ids", None)
    check_equal(out, gmo.mcts(roots, 32, 0, gmo.EVAL_HASH, seed=9, uids=uids, nthreads=8))


def same(a, b, keys=("visits", "q", "pi", "n_nodes")):
    return all(torch.equal(a[k].view(torch.int64) if a[k].dtype == torch.float64 else a[k],
                           b[k].view(torch.int64) if b[k].dtype == torch.float64 else b[k]) for k in keys)


@pytest.mark.parametrize("kernel", ["tc", "tc_acc"])
def test_fused_net_loop_equals_round_trips(model, kernel):
    """search_net = search_with(model.evaluate_states) bit for bit; direct, captured and replayed round graphs agree"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    model.set_kernel(kernel)
    L, h = model.eng.L, model.eng.h
    try:
        for n, pre_expand in ((200, False), (300, True)):
            roots = dev(cfg4_roots(n, seed=21 + n, plies=7))
            m = BatchedMCTS(model.eng, num_itr=48, gumbel=True, gumbel_considered=8)
            want = m.search_with(roots, model.evaluate_states, pre_expand=pre_expand)
            before = L.ccx_graph_replays(h)
            for _ in range(3):
                got = m.search_net(roots, pre_expand=pre_expand)
                assert same(want, got, ("visits", "q", "pi", "n_nodes", "action"))
            if not os.environ.get("CCX_NO_GRAPH"):
                assert L.ccx_graph_replays(h) - before == 2
    finally:
        model.set_kernel("tc")


def test_puct_gumbel_puct_gives_the_same_puct(model):
    from chinesecheckersagent_b200.engine import BatchedMCTS
    roots = dev(cfg4_roots(128, seed=3))
    puct = BatchedMCTS(model.eng, num_itr=40)
    a1 = puct.search_net(roots)
    g = BatchedMCTS(model.eng, num_itr=40, gumbel=True).search_net(roots)
    assert g["action"].min().item() >= 0
    a2 = puct.search_net(roots)
    assert same(a1, a2)
    a3 = puct.search_with(roots, model.evaluate_states)
    assert same(a1, a3)
    assert model.eng.L.ccx_mcts_pool_bytes(model.eng.h) > 0


def test_rejected_combinations(eng):
    from chinesecheckersagent_b200 import _lib
    from chinesecheckersagent_b200.engine import BatchedMCTS, _p
    roots = dev(cfg4_roots(4))
    for kw in (dict(leaves_per_round=4), dict(reuse_tree=True), dict(gumbel_considered=0), dict(gumbel_scale=-1.0)):
        with pytest.raises(ValueError):
            BatchedMCTS(eng, gumbel=True, **kw)
    m = BatchedMCTS(eng, num_itr=8, gumbel=True)
    with pytest.raises(ValueError):
        m.search(roots)
    with pytest.raises(ValueError):
        m.search_with(roots, oracle_evaluator(0), pre_expand=True, root_noise=torch.zeros((4, 128), dtype=torch.float64, device="cuda"))
    eng.call("ccx_mcts_set_gumbel", 1, 16, 1.0, 50.0, 0.1, 0)
    try:
        out = torch.empty((4, 294), dtype=torch.int32, device="cuda")
        assert eng.L.ccx_mcts_search(eng.h, 4, _p(roots), 0, 8, 3.5, 1.0, 0, None, 0, 0, _p(out), None, None, None) == -5
        assert eng.L.ccx_mcts_begin_reuse(eng.h, 4, _p(roots), 8, 0, -1, -1, 1, None, None, 0, 0, None) == -5
        assert eng.L.ccx_mcts_select_leaves(eng.h, 4, 4, 3.5, _p(out)) == -5
        assert eng.L.ccx_mcts_run_net_leaves(eng.h, 4, 8, 4, 3.5, None, 0, 0) == -5
    finally:
        eng.call("ccx_mcts_set_gumbel", 0, 1, 0.0, 0.0, 0.0, 0)
    assert eng.L.ccx_mcts_set_gumbel(eng.h, 1, 0, 1.0, 50.0, 0.1, 0) == -1
    with pytest.raises(_lib.CcxError):
        eng.call("ccx_mcts_set_gumbel", 1, 4, -1.0, 50.0, 0.1, 0)
    BatchedMCTS(eng, num_itr=4).search(roots)                      # the engine is back in PUCT mode


def test_inactive_trees_report_no_action(eng):
    from chinesecheckersagent_b200.engine import BatchedMCTS
    roots = cfg4_roots(8, seed=5)
    roots[4, :4] |= np.uint64(3 << 56)                             # finished games: inactive trees with min_ply_status
    out = BatchedMCTS(eng, num_itr=8, gumbel=True).search_with(dev(roots), oracle_evaluator(0), min_ply_status=True)
    a, nn, pi = out["action"].cpu().numpy(), out["n_nodes"].cpu().numpy(), out["pi"].cpu().numpy()
    assert np.all(a[:4] == -1) and np.all(nn[:4] == -2) and not pi[:4].any()
    assert np.all(a[4:] >= 0) and np.all(nn[4:] > 0)


def test_selfplay_is_deterministic_compaction_safe_and_well_formed(model):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay

    def run(compact):
        sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=256, seed=9, num_itr=16, max_iters=400, gumbel=True,
                             gumbel_considered=8)
        st = sp.play_games(300, compact=compact, compact_min=24)
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
    t = a[4]
    state = t["state"].cpu().numpy().view(np.uint64)
    full = np.zeros((8, state.shape[1]), dtype=np.uint64)
    full[:5] = state
    pi = t["pi_y"].cpu().numpy()
    assert np.all(pi >= 0) and np.allclose(pi.sum(1), 1.0, atol=1e-5)
    assert (pi > 0).sum(1).min() > 1                               # improved policies, not one-hot visit counts
    masks = orc.movegen(full)
    for i in range(0, pi.shape[0], max(1, pi.shape[0] // 200)):
        for act in np.nonzero(pi[i])[0]:
            cid, off = divmod(int(act), 49)
            assert (int(masks[cid, i]) >> ((off // 7) * 8 + off % 7)) & 1


def test_selfplay_plays_the_searched_action(model):
    from chinesecheckersagent_b200.config import INITIAL_RANDOM_MOVES
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=64, seed=4, num_itr=8, max_iters=64, gumbel=True, log_moves=True)
    checked = 0
    for it in range(INITIAL_RANDOM_MOVES + 10):
        sp.step()
        log = sp.move_log.view(sp.max_iters, sp.n)[it].cpu().numpy().astype(np.int64)
        act = sp.action.cpu().numpy()
        mcts = ((log >> 25) & 1).astype(bool) & ((log >> 24) & 1).astype(bool)
        for g in np.nonzero(mcts)[0]:
            frm, to = log[g] & 0xFF, (log[g] >> 8) & 0xFF
            assert act[g] >= 0 and (act[g] % 49) == (to >> 3) * 7 + (to & 7)
            checked += 1
    assert checked > 0


def test_arena_gumbel_against_puct(model):
    from chinesecheckersagent_b200.arena import BatchedArena
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)
    res = BatchedArena(model, other, 16, seed=3, num_itr=(16, 24), gumbel=(True, False)).play(max_plies=300)
    assert res["games"] == 16 and res["p1_wins"] + res["p2_wins"] > 0 and res["overflowed"] == 0
    again = BatchedArena(model, other, 16, seed=3, num_itr=(16, 24), gumbel=(True, False)).play(max_plies=300)
    assert res == again
