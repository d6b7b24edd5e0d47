"""GPU tests of per-tree search budgets (include/ccx.h, ccx_mcts_begin_budget) and self-play playout cap randomization
(ccx_selfplay_playout_cap, BatchedSelfPlay full_search_prob): every budgeted tree ends bit for bit like its unbudgeted
counterpart in every tie rule, symmetry mode and net kernel; the fused loop equals the round trips, with graph replay and the
two-stream split; self-play at p = 1 is the cap off, the draw follows the host rule, and compaction, two nets and resignation
carry the cap through."""
import os

import numpy as np
import pytest
import torch

import oracle as orc
import playout_cap_ref as pc
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

WEIGHTS = os.path.join(GOLDEN, "good_model_weights.npz")
SEED = 0x5EED0000CAFE1234
CPUCT = 3.5
ERR_UNSUPPORTED = -5


@pytest.fixture(scope="module")
def model():
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    e = Engine(0)
    m = ResidualCNN(engine=e).load_weights(WEIGHTS)
    yield m
    e.close()


def dev(a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint64:
        a = a.view(np.int64)
    return torch.from_numpy(a).cuda()


def roots_after(n, seed, plies):
    st, _, _ = orc.step_random(orc.start_states(n), seed, 0, plies, nthreads=8)
    return st


def mixed_roots(n, seed):
    """openings (5 plies: inactive under min_ply = 6), mid-games and long random games (many terminal leaves near the end)"""
    a = roots_after(n // 3, seed, 5)
    b = roots_after(n // 3, seed + 1, 30)
    c = roots_after(n - 2 * (n // 3), seed + 2, 160)
    return dev(np.concatenate([a, b, c], axis=1))


def search(model, roots, num_itr, rounds, budget=None, noise=None, ties=0, fused=True, min_ply=-1):
    """one search through the C calls: begin (with or without budget), `rounds` rounds fused or as round trips, finalize"""
    from chinesecheckersagent_b200.engine import _p
    e, n = model.eng, roots.shape[1]
    e.call("ccx_mcts_set_tiebreak", ties, SEED, 1000)
    if budget is None:
        e.call("ccx_mcts_begin", n, _p(roots), num_itr, 0, min_ply, -1)
    else:
        e.call("ccx_mcts_begin_budget", n, _p(roots), num_itr, 0, min_ply, -1, _p(budget))
    stride = 128 if noise is not None else 0
    if fused:
        e.call("ccx_mcts_run_net", n, rounds, CPUCT, _p(noise), stride, 1)
    else:
        leaf = e.empty((5, n), torch.int64)
        for r in range(rounds):
            e.call("ccx_mcts_select", n, CPUCT, _p(leaf))
            p, v = model.evaluate_states(leaf)
            nz = noise if r == 0 else None
            e.call("ccx_mcts_expand_backup", n, _p(p), _p(v), _p(nz), stride if nz is not None else 0, 1)
    visits, q, nodes = e.empty((n, 294), torch.int32), e.empty((n, 294), torch.float64), e.empty((n,), torch.int32)
    e.call("ccx_mcts_finalize", n, 1.0, _p(visits), None, _p(q), _p(nodes))
    return visits, q.view(torch.int64), nodes


def rows_equal(a, b, idx):
    return all(torch.equal(x[idx], y[idx]) for x, y in zip(a, b))


@pytest.mark.parametrize("kernel", ["tc_acc", "tc", "simt"])
@pytest.mark.parametrize("sym", ["off", "random", "mean"])
@pytest.mark.parametrize("ties", [0, 1])
def test_budget_rule(model, kernel, sym, ties):
    """tree i with b_i == S ends as the unbudgeted S-round search with the same noise, with b_i < S as a b_i-round search
    without noise: visits, Q bits and node counts"""
    S, n = 24, 501
    model.set_kernel(kernel)
    model.set_symmetry(sym, SEED)
    try:
        roots = mixed_roots(n, seed=ties + 3)
        g = torch.Generator(device="cpu").manual_seed(ties * 7 + len(kernel))
        levels = torch.tensor([S, S, 17, 9, 5, 1, 0, S + 40, -3], dtype=torch.int32)
        budget = levels[torch.randint(0, len(levels), (n,), generator=g)].cuda()
        noise = torch.rand((n, 128), dtype=torch.float64, device="cuda")
        got = search(model, roots, S, S, budget=budget, noise=noise, ties=ties, min_ply=6)
        eff = budget.clamp(0, S)
        assert int((got[2] == -2).sum()) >= n // 3 - 1            # the openings are inactive
        for b in sorted(set(eff.tolist())):
            want = search(model, roots, S, b, noise=noise if b == S else None, ties=ties, min_ply=6)
            idx = torch.nonzero(eff == b).flatten()
            assert rows_equal(got, want, idx), (kernel, sym, ties, b)
            if b < S:
                assert bool((want[0][idx].sum(1) <= b).all())
    finally:
        model.set_symmetry("off")
        model.set_kernel("tc_acc")


@pytest.mark.parametrize("ties", [0, 1])
def test_full_budgets_are_todays_search(model, ties):
    S, n = 30, 300
    roots = mixed_roots(n, seed=11)
    noise = torch.rand((n, 128), dtype=torch.float64, device="cuda")
    full = torch.full((n,), S, dtype=torch.int32, device="cuda")
    want = search(model, roots, S, S, noise=noise, ties=ties)
    for fused in (True, False):
        got = search(model, roots, S, S, budget=full, noise=noise, ties=ties, fused=fused)
        assert rows_equal(got, want, slice(None))


def same(a, b):
    return all(torch.equal(a[k].view(torch.int64) if a[k].dtype == torch.float64 else a[k],
                           b[k].view(torch.int64) if b[k].dtype == torch.float64 else b[k]) for k in ("visits", "q", "pi", "n_nodes"))


def budgets(n, full, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    fast = torch.randint(1, full, (n,), generator=g, dtype=torch.int32)
    return torch.where(torch.rand((n,), generator=g) < 0.3, torch.full_like(fast, full), fast).cuda()


def test_fused_equals_round_trips_and_graph_replay(model):
    from chinesecheckersagent_b200.engine import BatchedMCTS
    L, h = model.eng.L, model.eng.h
    n, S = 250, 40
    roots = mixed_roots(n, seed=21)
    nz = torch.rand((n, 128), dtype=torch.float64, device="cuda")
    m = BatchedMCTS(model.eng, num_itr=S, random_ties=True, tie_seed=5)
    kw = dict(pre_expand=True, root_noise=nz)
    b1 = budgets(n, S + 1, 1)
    want = m.search_with(roots, model.evaluate_states, budget=b1, **kw)
    before = L.ccx_graph_replays(h)
    for _ in range(3):                                   # direct, captured, replayed
        assert same(want, m.search_net(roots, budget=b1, **kw))
    if not os.environ.get("CCX_NO_GRAPH"):
        assert L.ccx_graph_replays(h) - before == 2
    # other budget contents at the same address: the replay follows them
    b1.copy_(budgets(n, S + 1, 2))
    before = L.ccx_graph_replays(h)
    assert same(m.search_with(roots, model.evaluate_states, budget=b1, **kw), m.search_net(roots, budget=b1, **kw))
    if not os.environ.get("CCX_NO_GRAPH"):
        assert L.ccx_graph_replays(h) - before == 1
    # an unbudgeted search after the budgeted one does not replay its graph, nor the reverse
    plain = m.search_with(roots, model.evaluate_states, **kw)
    before = L.ccx_graph_replays(h)
    assert same(plain, m.search_net(roots, **kw))
    assert L.ccx_graph_replays(h) == before
    assert same(m.search_with(roots, model.evaluate_states, budget=b1, **kw), m.search_net(roots, budget=b1, **kw))
    assert L.ccx_graph_replays(h) == before


def test_two_stream_split_with_budgets(model):
    """16,403 trees in the accurate mode: two ragged halves on two streams, equal to the round trips"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    n, S = 16403, 9
    roots = dev(roots_after(n, seed=77, plies=12))
    nz = torch.rand((n, 128), dtype=torch.float64, device="cuda")
    m = BatchedMCTS(model.eng, num_itr=S)
    b = budgets(n, S + 1, 3)
    want = m.search_with(roots, model.evaluate_states, pre_expand=True, root_noise=nz, budget=b)
    got = m.search_net(roots, pre_expand=True, root_noise=nz, budget=b)
    assert same(want, got)


def sp_of(model, **kw):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    return BatchedSelfPlay(model.eng, model.evaluate_states, **kw)


def drain_result(sp, games, **kw):
    st = sp.play_games(games, **kw)
    t = sp.collect()
    return st, {k: v.clone() for k, v in t.items()}, sp.env.state.clone()


@pytest.mark.parametrize("mode,trees", [("off", 16403), ("mean", 8203)])
def test_two_stream_split_with_budgets_all_kernels(model, mode, trees):
    """the 16-bit mode at the split threshold (the mean evaluates two rows per tree): each half packs its rows from its own start"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    model.set_kernel("tc")
    model.set_symmetry(mode, SEED)
    try:
        roots = dev(roots_after(trees, seed=trees, plies=10))
        m = BatchedMCTS(model.eng, num_itr=9, random_ties=True)
        b = budgets(trees, 10, 4)
        nz = torch.rand((trees, 128), dtype=torch.float64, device="cuda")
        want = m.search_with(roots, model.evaluate_states, pre_expand=True, root_noise=nz, budget=b)
        got = m.search_net(roots, pre_expand=True, root_noise=nz, budget=b)
        assert same(want, got)
    finally:
        model.set_symmetry("off")
        model.set_kernel("tc_acc")


def test_budgeted_search_leaves_the_engine_usable(model):
    """after cap self-play on an engine, a tree-reuse search (fresh: nothing is carried from budgeted trees) and an in-kernel
    search run as on a fresh engine"""
    from chinesecheckersagent_b200.engine import BatchedMCTS, Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    n = 64
    roots = mixed_roots(n, seed=5)
    sp = sp_of(model, n_slots=n, num_itr=10, max_iters=64, seed=3, full_search_prob=0.5, fast_itr=3)
    for _ in range(12):
        sp.step()
    eng2 = Engine(0)
    try:
        m2 = ResidualCNN(engine=eng2).load_weights(WEIGHTS)
        for mk in (lambda e: BatchedMCTS(e, num_itr=16, reuse_tree=True),):
            got = mk(model.eng).search_net(roots)
            want = mk(m2.eng).search_net(roots)
            assert same(got, want) and torch.equal(got["reused"], want["reused"]) and not bool((got["reused"] > 0).any())
        sp.step()
        a = BatchedMCTS(model.eng, num_itr=32).search(roots)
        b = BatchedMCTS(m2.eng, num_itr=32).search(roots)
        assert same(a, b)
    finally:
        eng2.close()


def test_fast_itr_equal_to_num_itr_still_drops_fast_records(model):
    kw = dict(n_slots=96, num_itr=8, max_iters=400, seed=29)
    a = drain_result(sp_of(model, **kw), 120)
    b = drain_result(sp_of(model, full_search_prob=0.5, fast_itr=8, **kw), 120)
    assert b[0]["fast_searches"] > 0 and 0 < b[0]["records"] < a[0]["records"]


@pytest.mark.parametrize("fused", [True, False])
def test_selfplay_cap_at_one_is_invisible(model, fused):
    kw = dict(n_slots=96, num_itr=12, max_iters=400, seed=23, fused=fused)
    a = drain_result(sp_of(model, **kw), 160)
    b = drain_result(sp_of(model, full_search_prob=1.0, fast_itr=4, **kw), 160)
    assert a[0]["records"] > 0
    assert {k: a[0][k] for k in a[0]} == {k: b[0][k] for k in a[0]}
    assert b[0]["fast_searches"] == 0 and b[0]["full_searches"] >= b[0]["records"]
    assert torch.equal(a[2], b[2])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k
    c = drain_result(sp_of(model, full_search_prob=0.0, fast_itr=4, **kw), 160)
    # games still finish; `games` counts the games that left a record, so none
    assert c[0]["records"] == 0 and c[0]["games"] == 0 and c[0]["p1_wins"] + c[0]["p2_wins"] > 0 and c[0]["unfinished"] == 0
    assert c[0]["full_searches"] == 0 and c[0]["fast_searches"] > 0


def test_selfplay_draw_is_the_host_rule(model):
    """kept records = the full-drawn searched plies of the kept games; full + fast = searched plies"""
    n, iters, p, seed = 192, 300, 0.3, 31
    sp = sp_of(model, n_slots=n, num_itr=12, max_iters=iters, seed=seed, log_moves=True, full_search_prob=p, fast_itr=3)
    plies = []
    for _ in range(iters):
        plies.append(((sp.env.state[4] >> 32) & 0xFFFF).cpu().numpy())
        sp.step(restart=False)
        if sp.running() == 0:
            break
    k = len(plies)
    log = sp.move_log.view(iters, n)[:k].cpu().numpy().astype(np.int64)
    flags = (sp.rec_flag.view(iters, n)[:k] & 0xF).cpu().numpy()
    final = (sp.env.state[4] >> 56).cpu().numpy()
    searched = ((log >> 24) & 1).astype(bool) & ((log >> 25) & 1).astype(bool)
    st = sp.stats()
    assert st["full_searches"] + st["fast_searches"] == int(searched.sum())
    kept = 0
    for s in range(n):
        its = np.nonzero(searched[:, s])[0]
        full = np.array([pc.full_search(seed, s, 0, plies[t][s], p)[0] for t in its], dtype=bool)
        if final[s] in (1, 2):
            assert np.array_equal(np.isin(flags[its, s], (2, 3)), full), s
            kept += int(full.sum())
        assert not np.any(flags[its[~full], s])
    assert st["records"] == kept > 0
    assert 0.15 < st["full_searches"] / (st["full_searches"] + st["fast_searches"]) < 0.45


def test_selfplay_cap_compaction_two_nets_resignation(model):
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN

    def run(compact):
        sp = sp_of(model, n_slots=320, seed=9, num_itr=10, max_iters=400, full_search_prob=0.25, fast_itr=3)
        st = sp.play_games(400, compact=compact, compact_min=24)
        t = sp.collect()
        key = np.vstack([t["state"].cpu().numpy(), t["v_y"].cpu().numpy()[None].astype(np.int64),
                         (t["pi_y"].double() * torch.arange(1, 295, device=t["pi_y"].device)).sum(1).mul(1e6).round().long().cpu().numpy()[None]])
        order = np.lexsort(key)
        return st, t["board_x"].cpu().numpy()[order], t["pi_y"].cpu().numpy()[order], t["v_y"].cpu().numpy()[order], sp.n
    a, b = run(False), run(True)
    assert b[0]["compactions"] >= 1 and a[0]["compactions"] == 0 and b[4] < a[4]
    assert {k: v for k, v in a[0].items() if k != "compactions"} == {k: v for k, v in b[0].items() if k != "compactions"}
    assert a[1].shape[0] == a[0]["records"] > 0
    for x, y in zip(a[1:4], b[1:4]):
        assert np.array_equal(x, y)

    eng2 = Engine(0)
    try:
        m2 = ResidualCNN(engine=eng2).load_weights(WEIGHTS)
        kw = dict(n_slots=96, num_itr=12, max_iters=120, seed=13, log_moves=True, full_search_prob=0.4, fast_itr=5)
        x = sp_of(model, **kw)
        x.run(iters=120)
        y = sp_of(model, opponent=m2, **kw)
        y.run(iters=120)
        assert torch.equal(x.move_log, y.move_log) and torch.equal(x.rec_visits, y.rec_visits) and torch.equal(x.rec_flag, y.rec_flag)
        assert torch.equal(x.env.state, y.env.state) and x.stats() == y.stats() and x.stats()["fast_searches"] > 0
    finally:
        eng2.close()

    r = sp_of(model, n_slots=128, num_itr=10, max_iters=400, seed=19, full_search_prob=0.3, fast_itr=3, resign_threshold=-0.2,
              resign_plies=2, resign_probe=0.2)
    st = r.play_games(200)
    assert st["games_started"] == 200 and st["unfinished"] == 0
    assert 0 < st["records"] <= st["full_searches"] and st["fast_searches"] > 0
    assert st["probe_games"] <= st["p1_wins"] + st["p2_wins"]


def test_arguments(model):
    from chinesecheckersagent_b200.engine import BatchedMCTS, _p
    for bad in (dict(full_search_prob=0.5, leaves_per_round=2), dict(full_search_prob=0.5, gumbel=True),
                dict(full_search_prob=0.5, reuse_tree=True), dict(full_search_prob=1.5), dict(full_search_prob=-0.1),
                dict(full_search_prob=0.5, fast_itr=0), dict(full_search_prob=0.5, fast_itr=13)):
        with pytest.raises(ValueError):
            sp_of(model, n_slots=8, num_itr=12, **bad)
    n = 16
    roots = mixed_roots(n, seed=2)
    bud = torch.full((n,), 5, dtype=torch.int32, device="cuda")
    for kw in (dict(leaves_per_round=2), dict(gumbel=True), dict(reuse_tree=True)):
        with pytest.raises(ValueError):
            BatchedMCTS(model.eng, num_itr=8, **kw).search_net(roots, budget=bud)
    with pytest.raises(ValueError):
        BatchedMCTS(model.eng, num_itr=8).search_net(roots, budget=bud.long())
    e = model.eng
    L, h = e.L, e.h
    leaf = e.empty((5, n * 4), torch.int64)
    vis = e.empty((n, 294), torch.int32)
    assert L.ccx_mcts_begin_budget(h, n, _p(roots), 8, 0, -1, -1, _p(bud)) == 0
    assert L.ccx_mcts_select_leaves(h, n, 4, CPUCT, _p(leaf)) == ERR_UNSUPPORTED
    assert L.ccx_mcts_leaf_budget(h, n, 4, 8) == ERR_UNSUPPORTED
    assert L.ccx_mcts_run_net_leaves(h, n, 8, 4, CPUCT, None, 0, 0) == ERR_UNSUPPORTED
    assert L.ccx_mcts_set_gumbel(h, 1, 4, 1.0, 50.0, 0.1, 0) == 0
    try:
        assert L.ccx_mcts_run_net(h, n, 8, CPUCT, None, 0, 0) == ERR_UNSUPPORTED
        assert L.ccx_mcts_begin_budget(h, n, _p(roots), 8, 0, -1, -1, _p(bud)) == ERR_UNSUPPORTED
    finally:
        assert L.ccx_mcts_set_gumbel(h, 0, 1, 0.0, 0.0, 0.0, 0) == 0
    # new searches of every kind start without budgets
    reused = e.empty((n,), torch.int32)
    assert L.ccx_mcts_begin_budget(h, n, _p(roots), 8, 0, -1, -1, _p(bud)) == 0
    assert L.ccx_mcts_search(h, n, _p(roots), 0, 8, CPUCT, 1.0, 0, None, 0, 0, _p(vis), None, None, None) == 0
    assert L.ccx_mcts_select_leaves(h, n, 4, CPUCT, _p(leaf)) == 0
    assert L.ccx_mcts_begin_budget(h, n, _p(roots), 8, 0, -1, -1, _p(bud)) == 0
    assert L.ccx_mcts_begin_reuse(h, n, _p(roots), 8, 0, -1, -1, 1, None, None, 0, 0, _p(reused)) == 0
    assert not bool((reused > 0).any())
    assert L.ccx_mcts_select_leaves(h, n, 4, CPUCT, _p(leaf)) == 0
    torch.cuda.synchronize()
