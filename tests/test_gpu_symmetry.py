"""GPU tests of the mirror-symmetric net evaluation (include/ccx.h ccx_net_set_symmetry, ResidualCNN.set_symmetry):
ccx_net_eval bit for bit against the restatement built from the raw forward pass on explicitly mirrored planes
(tests/symmetry_ref.py), mode 0 unchanged, the fused loops (one-leaf PUCT, leaf-parallel, Gumbel) equal to the round trips
with tree reuse, graph replay and the two-stream split, mode switches between searches, self-play and the arena."""
import os

import numpy as np
import pytest
import torch

import oracle as orc
import symmetry_ref as sr
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

WEIGHTS = os.path.join(GOLDEN, "good_model_weights.npz")
SEED = 0x5EED0000CAFE1234


@pytest.fixture(scope="module")
def model():
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    return ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)


@pytest.fixture(scope="module")
def other():
    """the same net in a second engine (its own handle and trees)"""
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    return ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS)


def dev(a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint64:
        a = a.view(np.int64)
    return torch.from_numpy(a).cuda()


def roots_after(n, seed, plies=6):
    st, _, _ = orc.step_random(orc.start_states(n), seed, 0, plies, nthreads=8)
    return st


def mixed_states(n, seed):
    """random play from the start, randomised placements and mid-game positions"""
    if n < 3:
        return roots_after(n, seed, 5)
    a = roots_after(n // 3, seed, 5)
    b, _, _ = orc.step_random(orc.random_states(n // 3, seed + 1), seed + 2, 0, 3, nthreads=8)
    c = roots_after(n - 2 * (n // 3), seed + 3, 41)
    return np.ascontiguousarray(np.concatenate([a, b, c], axis=1))


def play(st, acts):
    acts = np.asarray(acts, dtype=np.int64)
    side = (st[4] >> np.uint64(48)) & np.uint64(1)
    cells = np.where(side == 1, st[3], st[2])
    cid, off = acts // 49, acts % 49
    frm = ((cells >> (np.uint64(8) * cid.astype(np.uint64))) & np.uint64(0xFF)).astype(np.uint8)
    to = ((off // 7) * 8 + off % 7).astype(np.uint8)
    return orc.apply(st, frm, to)[0]


def same(a, b, keys=("visits", "q", "pi", "n_nodes")):
    return all(torch.equal(a[k].view(torch.int64) if a[k].dtype == torch.float64 else a[k],
                           b[k].view(torch.int64) if b[k].dtype == torch.float64 else b[k]) for k in keys)


def raw_eval(model, planes):
    """ccx_net_forward_u8 + ccx_softmax_f64 on an explicit batch of planes: (p rows, v rows) float64 on the host"""
    e = model.eng
    x = dev(planes.astype(np.uint8))
    n = x.shape[0]
    logits, value = e.empty((n, 294), torch.float32), e.empty((n,), torch.float32)
    p, v = e.empty((n, 294), torch.float64), e.empty((n,), torch.float64)
    e.call("ccx_net_forward_u8", n, x.data_ptr(), logits.data_ptr(), value.data_ptr())
    e.call("ccx_softmax_f64", n, logits.data_ptr(), value.data_ptr(), p.data_ptr(), v.data_ptr())
    return p.cpu().numpy(), v.cpu().numpy()


@pytest.mark.parametrize("kernel", ["simt", "tc", "tc_acc"])
@pytest.mark.parametrize("mode", ["random", "mean"])
def test_net_eval_matches_the_restatement(model, kernel, mode):
    model.set_kernel(kernel)
    try:
        for n in (1, 77, 301):
            st = mixed_states(n, seed=n * 7 + len(kernel))
            flags = sr.mirrored(st, SEED)
            assert n < 10 or 0 < flags.sum() < n
            model.set_symmetry(mode, SEED)
            p, v = model.evaluate_states(dev(st[:5]))
            model.set_symmetry("off")
            rows = sr.net_rows(orc.encode(st), sr.MODES[mode], flags)
            want_p, want_v = sr.combine(*raw_eval(model, rows), sr.MODES[mode], flags)
            assert np.array_equal(p.cpu().numpy().view(np.uint64), want_p.view(np.uint64))
            assert np.array_equal(v.cpu().numpy().view(np.uint64), want_v.view(np.uint64))
    finally:
        model.set_symmetry("off")
        model.set_kernel("tc_acc")


def test_mode_off_is_the_untouched_handle(model, other):
    """a handle that went through random and mean and back to off evaluates and searches as one that never called the setter"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    st = dev(mixed_states(150, seed=5)[:5])
    roots = dev(roots_after(150, seed=6))
    model.set_symmetry("random", 1)
    model.set_symmetry("mean", 2)
    mean_p, _ = model.evaluate_states(st)
    model.set_symmetry("off", 3)
    p, v = model.evaluate_states(st)
    q, w = other.evaluate_states(st)
    assert torch.equal(p, q) and torch.equal(v, w) and not torch.equal(p, mean_p)
    a = BatchedMCTS(model.eng, num_itr=24).search_net(roots)
    b = BatchedMCTS(other.eng, num_itr=24).search_net(roots)
    assert same(a, b)
    # the raw forward pass and softmax are not symmetrised
    planes = torch.from_numpy(orc.encode(mixed_states(40, seed=8))).cuda()
    base = model.predict_batch(planes)
    model.set_symmetry("mean")
    try:
        again = model.predict_batch(planes)
        assert torch.equal(base[0], again[0]) and torch.equal(base[1], again[1])
    finally:
        model.set_symmetry("off")


def test_bad_mode_is_refused(model):
    L, h = model.eng.L, model.eng.h
    assert L.ccx_net_set_symmetry(h, 3, 0) == -1 and L.ccx_net_set_symmetry(h, -1, 0) == -1
    with pytest.raises(ValueError):
        model.set_symmetry("both")


FUSED = [  # (leaves, gumbel, random_ties, root noise)
    (1, False, False, True), (1, False, True, False), (4, False, True, True), (16, False, False, False), (1, True, False, False),
]


@pytest.mark.parametrize("mode", ["random", "mean"])
@pytest.mark.parametrize("leaves,gumbel,ties,noise", FUSED)
def test_fused_loop_equals_round_trips(model, mode, leaves, gumbel, ties, noise):
    """search_net = search_with(model.evaluate_states) bit for bit; the direct run, the captured and the replayed graph agree"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    L, h = model.eng.L, model.eng.h
    model.set_symmetry(mode, SEED)
    try:
        for n in (200, 67):
            roots = dev(roots_after(n, seed=n + leaves))
            nz = torch.rand((n, 128), dtype=torch.float64, device="cuda") if noise else None
            sims = 120 if leaves == 16 else 40                # at least 8 launched rounds: the loop is graph-cached
            m = BatchedMCTS(model.eng, num_itr=sims, leaves_per_round=leaves, random_ties=ties, tie_seed=0xC0FFEE, tie_uid0=100,
                            gumbel=gumbel, gumbel_considered=8)
            kw = dict(pre_expand=noise, root_noise=nz)
            want = m.search_with(roots, model.evaluate_states, **kw)
            before = L.ccx_graph_replays(h)
            for _ in range(3):
                got = m.search_net(roots, **kw)
                assert same(want, got, ("visits", "q", "pi", "n_nodes") + (("action",) if gumbel else ()))
            if not os.environ.get("CCX_NO_GRAPH"):
                assert L.ccx_graph_replays(h) - before == 2
    finally:
        model.set_symmetry("off")


@pytest.mark.parametrize("mode", ["random", "mean"])
@pytest.mark.parametrize("leaves", [1, 4])
def test_fused_loop_with_reuse_equals_round_trips(model, other, mode, leaves):
    from chinesecheckersagent_b200.engine import BatchedMCTS
    model.set_symmetry(mode, SEED)
    other.set_symmetry(mode, SEED)
    try:
        n = 160
        st = roots_after(n, seed=12)
        noise = torch.rand((n, 128), dtype=torch.float64, device="cuda")
        a = BatchedMCTS(model.eng, num_itr=24, leaves_per_round=leaves, reuse_tree=True)
        b = BatchedMCTS(other.eng, num_itr=24, leaves_per_round=leaves, reuse_tree=True)
        for ply in range(4):
            got = a.search_net(dev(st), pre_expand=True, root_noise=noise)
            want = b.search_with(dev(st), other.evaluate_states, pre_expand=True, root_noise=noise)
            assert same(want, got) and torch.equal(want["reused"], got["reused"])
            if ply:
                assert int((got["reused"] == 1).sum()) > n // 2
            st = play(st, got["visits"].argmax(1).cpu().numpy())
    finally:
        model.set_symmetry("off")
        other.set_symmetry("off")


@pytest.mark.parametrize("mode,trees,leaves", [("mean", 4096, 1), ("random", 8192, 1), ("mean", 1024, 4)])
def test_two_stream_split_equals_round_trips(model, mode, trees, leaves):
    """batches at the split threshold (8,192 net rows in the 16-bit mode; the mean mode evaluates two rows per leaf): the
    fused loop runs as two halves on two streams and still equals the round trips"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    model.set_kernel("tc")
    model.set_symmetry(mode, SEED)
    try:
        roots = dev(roots_after(trees, seed=trees + leaves))
        m = BatchedMCTS(model.eng, num_itr=9, leaves_per_round=leaves)
        want = m.search_with(roots, model.evaluate_states)
        got = m.search_net(roots)
        assert same(want, got)
    finally:
        model.set_symmetry("off")
        model.set_kernel("tc_acc")


def test_mode_switches_between_searches(model):
    """A / B / A on one handle: each search gets its own mode's result; a carried tree is not reused across a switch"""
    from chinesecheckersagent_b200.engine import BatchedMCTS
    roots = dev(roots_after(128, seed=31))
    m = BatchedMCTS(model.eng, num_itr=32)
    try:
        model.set_symmetry("random", SEED)
        a1 = m.search_net(roots)
        model.set_symmetry("mean", SEED)
        b1 = m.search_net(roots)
        model.set_symmetry("random", SEED)
        a2 = m.search_net(roots)
        model.set_symmetry("random", SEED + 1)
        c1 = m.search_net(roots)
        model.set_symmetry("off")
        o1 = m.search_net(roots)
        assert same(a1, a2) and not same(a1, b1) and not same(a1, o1) and not same(b1, o1) and not same(a1, c1)
        model.set_symmetry("random", SEED)
        assert same(a1, m.search_with(roots, model.evaluate_states))
        # tree reuse: a switch starts every tree fresh, no switch carries
        r = BatchedMCTS(model.eng, num_itr=32, reuse_tree=True)
        st = roots_after(128, seed=31)
        first = r.search_net(dev(st))
        st = play(st, first["visits"].argmax(1).cpu().numpy())
        model.set_symmetry("mean", SEED)
        fresh = r.search_net(dev(st))
        assert not fresh["reused"].any()
        assert same(fresh, BatchedMCTS(model.eng, num_itr=32).search_net(dev(st)))
        st2 = play(st, fresh["visits"].argmax(1).cpu().numpy())
        r.search_net(dev(st))
        carried = r.search_net(dev(st2))
        assert int((carried["reused"] == 1).sum()) > 64
    finally:
        model.set_symmetry("off")


def run_selfplay(model, compact):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=256, seed=9, num_itr=16, max_iters=400)
    st = sp.play_games(300, compact=compact, compact_min=24)
    t = sp.collect()
    key = np.vstack([t["state"].cpu().numpy(), t["v_y"].cpu().numpy()[None].astype(np.int64),
                     (t["pi_y"].double() * torch.arange(1, 295, device=t["pi_y"].device)).sum(1).mul(1e6).round().long().cpu().numpy()[None]])
    order = np.lexsort(key)
    return st, t["board_x"].cpu().numpy()[order], t["pi_y"].cpu().numpy()[order], t["v_y"].cpu().numpy()[order]


def test_selfplay_mean_is_deterministic_and_compaction_safe(model):
    model.set_symmetry("mean")
    try:
        a, c = run_selfplay(model, False), run_selfplay(model, True)
    finally:
        model.set_symmetry("off")
    assert a[0]["records"] > 0 and a[0]["games"] > 0 and c[0]["compactions"] >= 1
    for k in ("plies", "p1_wins", "p2_wins", "records", "games", "iterations"):
        assert a[0][k] == c[0][k], k
    for i in (1, 2, 3):
        assert np.array_equal(a[i], c[i])


def test_arena_with_a_mode_per_side(model, other):
    from chinesecheckersagent_b200.arena import BatchedArena
    model.set_symmetry("random", SEED)
    other.set_symmetry("mean")
    try:
        res = BatchedArena(model, other, 16, seed=3, num_itr=16).play(max_plies=300)
        assert res["games"] == 16 and res["p1_wins"] + res["p2_wins"] > 0 and res["overflowed"] == 0
        assert res == BatchedArena(model, other, 16, seed=3, num_itr=16).play(max_plies=300)
        other.set_symmetry("off")
        assert res != BatchedArena(model, other, 16, seed=3, num_itr=16).play(max_plies=300)
    finally:
        model.set_symmetry("off")
        other.set_symmetry("off")
