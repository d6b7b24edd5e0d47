"""GPU tests of tree reuse (include/ccx.h ccx_mcts_begin_reuse): multi-ply searches bit for bit against the C oracle's
persistent trees (tests/reuse_oracle), the fused net loop equal to the round trips with its cached graph replayed across
plies, and self-play / the arena running with it."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle as orc
from conftest import GOLDEN

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "leaves_oracle"))
import leaves_oracle as lvo  # noqa: E402
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "reuse_oracle"))
import reuse_oracle as rvo  # noqa: E402

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


def play(st, acts):
    """apply policy index acts[i] (checker id * 49 + destination r*7+c) to the side to move of every state"""
    acts = np.asarray(acts, dtype=np.int64)
    side = (st[4] >> np.uint64(48)) & np.uint64(1)
    cells = np.where(side == 1, st[3], st[2])
    cid, off = acts // 49, acts % 49
    frm = ((cells >> (np.uint64(8) * cid.astype(np.uint64))) & np.uint64(0xFF)).astype(np.uint8)
    to = ((off // 7) * 8 + off % 7).astype(np.uint8)
    return orc.apply(st, frm, to)[0]


def most_visited_reply(f, i, act):
    """the reply with the most visits below tree i's move `act` (the highest prior when none has a visit yet)"""
    N, _, P = f.child_stats(i, act)
    return N.argmax() if N.any() else P.argmax()


def oracle_evaluator(evaluator):
    def evaluate(leaf):
        st = np.zeros((8, leaf.shape[1]), dtype=np.uint64)
        st[:5] = leaf.cpu().numpy().view(np.uint64)
        p, v = lvo.eval_batch(orc.encode(st), evaluator)
        return dev(p), dev(v)
    return evaluate


def assert_same(out, want, reused_want):
    v, pi, q, nodes = want
    assert np.array_equal(out["visits"].cpu().numpy().astype(np.uint32), v)
    assert np.array_equal(out["q"].cpu().numpy().view(np.uint64), q.view(np.uint64))
    assert np.array_equal(out["pi"].cpu().numpy(), pi)
    assert np.array_equal(out["n_nodes"].cpu().numpy(), nodes)
    assert np.array_equal(out["reused"].cpu().numpy(), reused_want)


def same_search(a, b):
    return (torch.equal(a["visits"], b["visits"]) and torch.equal(a["q"].view(torch.int64), b["q"].view(torch.int64))
            and torch.equal(a["pi"].view(torch.int64), b["pi"].view(torch.int64)) and torch.equal(a["n_nodes"], b["n_nodes"]))


@pytest.mark.parametrize("leaves", [1, 4])
@pytest.mark.parametrize("ties", [None, (0xC0FFEE, 1000)])
@pytest.mark.parametrize("noise", [False, True])
def test_search_with_reuse_matches_the_oracle(eng, leaves, ties, noise):
    """six plies on 96 roots: fresh, depth 1, depth 2, depth 1 through a permuted prev with -1 / out-of-range entries, then
    unrelated and inactive roots mixed in; visits, pi, root Q bits, node counts and `reused` equal the oracle at every ply"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    n, num_itr, cpuct, carry = 96, 40, 1.5, 3
    st = cfg4_roots(n, seed=0x5EED2026 + leaves)
    rng = np.random.default_rng(leaves)
    kw = dict(random_ties=True, tie_seed=ties[0], tie_uid0=ties[1]) if ties else {}
    m = BatchedMCTS(eng, cpuct=cpuct, num_itr=num_itr, leaves_per_round=leaves, reuse_tree=True, reuse_carry=carry, **kw)
    f = rvo.Forest()
    depths = set()
    for ply in range(6):
        prev = None
        if ply == 3:
            perm = rng.permutation(n)
            st, prev = st[:, perm], perm.copy()
            prev[:4] = (-1, n, n + 7, 1 << 40)
        if ply == 4:
            other = cfg4_roots(n, seed=77)
            st[:, :8] = other[:, :8]                                    # no match
            st[4, 8:12] |= np.uint64(1 << 56)                           # finished games: inactive
        nz = rng.dirichlet(np.ones(128) * 0.3, size=n) if noise else None
        out = m.search_with(dev(st), oracle_evaluator(orc.EVAL_HASH), pre_expand=noise, root_noise=dev(nz) if noise else None,
                            prev=dev(prev) if prev is not None else None, min_ply_status=True)
        reused = f.begin(st, num_itr + 1, carry, prev=prev, noise=nz, min_ply=0)
        f.search(num_itr + int(noise), leaves, cpuct, orc.EVAL_HASH, noise=nz, ties=ties)
        stats = {}
        want = f.finalize(stats=stats)
        assert_same(out, want, reused)
        assert not stats["vl_left"].any()
        depths |= set(np.unique(reused).tolist())
        if ply == 0:
            assert not reused.any()
        if ply == 4:
            assert not reused[:8].any() and (reused[8:12] == -2).all()
        acts = want[0].argmax(1)
        if ply == 1:                                                    # the move and the reply the tree explored most
            reply = np.array([most_visited_reply(f, i, a) for i, a in enumerate(acts)])
            st = play(play(st, acts), reply)
        elif ply == 4:                                                  # the finished games stay where they are, running again
            moved = play(st, acts)
            moved[:, 8:12] = st[:, 8:12]
            moved[4, 8:12] &= ~np.uint64(0xFF << 56)
            st = moved
        else:
            st = play(st, acts)
    assert {0, 1, 2, -2} <= depths


def test_carry_limit_and_net_reload(model):
    """a carried root with more visits than carry (S + 1) falls back to a fresh tree, on the GPU as in the oracle; loading
    the net's weights again starts every tree fresh"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    e = model.eng
    n, E = 64, 20000
    st = cfg4_roots(n, seed=31)
    big = BatchedMCTS(e, num_itr=200, edges_per_tree=E, reuse_tree=True, reuse_carry=1)
    small = BatchedMCTS(e, num_itr=10, edges_per_tree=E, reuse_tree=True, reuse_carry=1)
    f = rvo.Forest()
    ev = oracle_evaluator(orc.EVAL_HASH)
    for mm, S in ((big, 201), (small, 11), (big, 201), (big, 201)):
        out = mm.search_with(dev(st), ev)
        reused = f.begin(st, S, 1, edges_per_tree=E)
        f.search(S - 1, 1, 3.5, orc.EVAL_HASH)
        want = f.finalize()
        assert_same(out, want, reused)
        if mm is small:
            assert (reused == 0).sum() > 8
        st = play(st, want[0].argmax(1))
    model.load_weights(WEIGHTS)                                         # ccx_net_load / ccx_net_load_tc: a new evaluator
    out = big.search_with(dev(st), ev)
    f.invalidate()
    reused = f.begin(st, 201, 1, edges_per_tree=E)
    f.search(200, 1, 3.5, orc.EVAL_HASH)
    assert_same(out, f.finalize(), reused)
    assert not reused.any()
    assert e.L.ccx_mcts_pool_bytes(e.h) > 0


@pytest.mark.parametrize("kernel", ["tc", "tc_acc"])
@pytest.mark.parametrize("leaves", [1, 4])
def test_fused_net_loop_with_reuse_equals_round_trips(model, kernel, leaves):
    """search_net with reuse = search_with(model.evaluate_states) with reuse, ply after ply (two engines with the same net,
    each carrying its own trees); the cached round graph keeps being replayed across plies"""
    from chinesecheckersagent_b200.engine import BatchedMCTS, Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)
    model.set_kernel(kernel)
    other.set_kernel(kernel)
    L, h = model.eng.L, model.eng.h
    try:
        n = 300
        st = cfg4_roots(n, seed=4)
        noise = torch.rand((n, 128), dtype=torch.float64, device="cuda")
        a = BatchedMCTS(model.eng, num_itr=32, leaves_per_round=leaves, reuse_tree=True)
        b = BatchedMCTS(other.eng, num_itr=32, leaves_per_round=leaves, reuse_tree=True)
        replays = []
        for ply in range(5):
            got = a.search_net(dev(st), pre_expand=True, root_noise=noise)
            want = b.search_with(dev(st), other.evaluate_states, pre_expand=True, root_noise=noise)
            assert same_search(want, got) and torch.equal(want["reused"], got["reused"])
            if ply:
                assert int((got["reused"] == 1).sum()) > n // 2
            replays.append(L.ccx_graph_replays(h))
            st = play(st, got["visits"].argmax(1).cpu().numpy())
        if not os.environ.get("CCX_NO_GRAPH"):
            assert replays[-1] - replays[1] == 3
    finally:
        model.set_kernel("tc")


def test_reuse_off_is_unchanged(model):
    """reuse_tree=False takes the plain begin: the same search as before, and `prev` is refused"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    roots = dev(cfg4_roots(64, seed=3))
    m = BatchedMCTS(model.eng, num_itr=24)
    a = m.search_net(roots)
    assert "reused" not in a
    r = BatchedMCTS(model.eng, num_itr=24, reuse_tree=True, reuse_carry=0).search_net(roots)
    assert same_search(a, r) and not r["reused"].any()
    with pytest.raises(ValueError):
        m.search_net(roots, prev=torch.arange(64, device="cuda"))


def run_selfplay(model, compact, seed=9, **kw):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=320, seed=seed, num_itr=16, max_iters=400, reuse_tree=True, **kw)
    st = sp.play_games(360, compact=compact, compact_min=24)
    t = sp.collect()
    key = np.vstack([t["state"].cpu().numpy(), t["v_y"].cpu().numpy()[None].astype(np.int64),
                     (t["pi_y"].double() * torch.arange(1, 295, device=t["pi_y"].device)).sum(1).mul(1e6).round().long().cpu().numpy()[None]])
    order = np.lexsort(key)
    return st, t["board_x"].cpu().numpy()[order], t["pi_y"].cpu().numpy()[order], t["v_y"].cpu().numpy()[order], t


@pytest.mark.parametrize("leaves", [1, 8])
def test_selfplay_with_reuse_is_deterministic_and_well_formed(model, leaves):
    a, b, c = (run_selfplay(model, False, leaves_per_round=leaves), run_selfplay(model, False, leaves_per_round=leaves),
               run_selfplay(model, True, leaves_per_round=leaves))
    assert a[0]["records"] > 0 and a[0]["games"] > 0
    for k in ("plies", "p1_wins", "p2_wins", "records", "games", "iterations", "reused_searches", "fresh_searches"):
        assert a[0][k] == b[0][k] == c[0][k], k
    for i in (1, 2, 3):
        assert np.array_equal(a[i], b[i]) and np.array_equal(a[i], c[i])
    assert c[0]["compactions"] >= 1
    # the env's successor states are the trees' child states: most searches after the opening continue a tree
    assert a[0]["reused_searches"] > a[0]["fresh_searches"]
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


def test_selfplay_reuse_rejects_an_opponent(model):
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)
    with pytest.raises(ValueError):
        BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=8, opponent=other, reuse_tree=True)


def test_arena_with_reuse_plays_every_game_to_the_end(model):
    from chinesecheckersagent_b200.arena import GREEDY, BatchedArena
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)
    for p1, p2, reuse in ((model, other, (True, False)), (model, GREEDY, True), (GREEDY, model, (False, True))):
        res = BatchedArena(p1, p2, 16, seed=3, num_itr=24, reuse_tree=reuse).play(max_plies=1000)
        assert res["games"] == 16 and res["unfinished"] == 0 and res["overflowed"] == 0
        again = BatchedArena(p1, p2, 16, seed=3, num_itr=24, reuse_tree=reuse).play(max_plies=1000)
        assert res == again
