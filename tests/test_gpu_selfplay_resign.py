"""GPU tests of opt-in self-play resignation (include/ccx.h, ccx_selfplay_resign): track-only runs change nothing, the kernel's
resign value is the host restatement's bit for bit, a resigned game is a prefix of its track-only counterpart, probe games and
calibration samples follow the host rule, and compaction, two nets and train.evolve carry it through."""
import math
import os

import numpy as np
import pytest
import torch

import resign_ref
from conftest import GOLDEN

pytestmark = pytest.mark.gpu
WEIGHTS = os.path.join(GOLDEN, "good_model_weights.npz")


@pytest.fixture(scope="module")
def model():
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    e = Engine(0)
    m = ResidualCNN(engine=e).load_weights(WEIGHTS)          # the accurate tensor-core mode (the default)
    assert m.kernel == "tc_acc"
    yield m
    e.close()


@pytest.fixture(scope="module")
def calib(model):
    """a threshold at which resignations happen: the 10 % false-positive suggestion of a track-only run"""
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=256, num_itr=12, max_iters=400, seed=4, resign_threshold=-1.0)
    st = sp.play_games(512)
    assert st["resign_samples_written"] == st["p1_wins"] + st["p2_wins"] > 50 and st["resigned_games"] == 0
    t = sp.suggest_resign_threshold(0.1)
    assert -1.0 < t < 1.0
    return t


def sp_of(model, **kw):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    return BatchedSelfPlay(model.eng, model.evaluate_states, **kw)


def drain_result(sp, games, **kw):
    st = sp.play_games(games, **kw)
    t = sp.collect()
    return st, {k: v.clone() for k, v in t.items()}, sp.env.state.clone()


BASE_KEYS = ("plies", "p1_wins", "p2_wins", "discarded_repetition", "discarded_no_progress", "discarded_overflow", "records", "games",
             "iterations", "unfinished", "compactions", "games_started")


@pytest.mark.parametrize("mode", ["puct", "leaves", "reuse", "gumbel", "mean"])
def test_track_only_is_invisible(model, mode):
    kw = dict(n_slots=96, num_itr=12, max_iters=400, seed=23)
    kw.update({"leaves": dict(leaves_per_round=4), "reuse": dict(reuse_tree=True), "gumbel": dict(gumbel=True)}.get(mode, {}))
    if mode == "mean":
        model.set_symmetry("mean", 5)
    try:
        a = drain_result(sp_of(model, **kw), 160)
        b = drain_result(sp_of(model, resign_threshold=-1.0, **kw), 160)
    finally:
        model.set_symmetry("off")
    assert a[0]["records"] > 0
    assert {k: a[0][k] for k in a[0]} == {k: b[0][k] for k in a[0]}
    assert "resigned_games" not in a[0] and b[0]["resigned_games"] == 0
    assert torch.equal(a[2], b[2])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k


def test_value_equals_the_host_restatement(model):
    """r written by the kernel == resign_ref.resign_value over the roots' edge order and N (ccx_mcts_get_root) and Q
    (ccx_mcts_finalize), bit for bit, over a few hundred self-play roots"""
    from chinesecheckersagent_b200.engine import _p
    e, n = model.eng, 64
    sp = sp_of(model, n_slots=n, num_itr=16, max_iters=64, seed=8, resign_threshold=-1.0)
    vis, q = e.empty((n, 294), torch.int32), e.empty((n, 294), torch.float64)
    ne, mv = e.empty((n,), torch.int32), e.empty((n, 128), torch.int16)
    N, W, P = e.empty((n, 128), torch.int32), e.empty((n, 128), torch.float64), e.empty((n, 128), torch.float64)
    checked = 0
    for it in range(40):
        sp.step()
        if it < 8 or it % 4:
            continue
        e.call("ccx_mcts_get_root", n, 128, _p(ne), _p(mv), _p(N), _p(W), _p(P))
        e.call("ccx_mcts_finalize", n, 1.0, _p(vis), None, _p(q), None)
        val, nodes = sp.resign_value.cpu().numpy(), sp.tree_nodes.cpu().numpy()
        ne_h, mv_h, N_h, q_h = ne.cpu().numpy(), mv.cpu().numpy().view(np.uint16), N.cpu().numpy(), q.cpu().numpy()
        for i in range(n):
            if nodes[i] < 0:
                assert math.isnan(val[i])
                continue
            k = int(ne_h[i])
            idx = [(m >> 8) * 49 + ((m & 0xFF) >> 3) * 7 + (m & 7) for m in mv_h[i, :k]]
            r = resign_ref.resign_value([int(x) for x in N_h[i, :k]], [float(q_h[i, a]) for a in idx])
            if math.isnan(r):
                assert math.isnan(val[i])
                continue
            assert np.float64(r).view(np.int64) == np.float64(val[i]).view(np.int64), (it, i, r, val[i])
            checked += 1
    assert checked >= 300


def logged_run(model, n, iters, **kw):
    """step() without restarts; per iteration the mover of every slot before the step, r and the status after it"""
    sp = sp_of(model, n_slots=n, max_iters=iters, **kw)
    movers, values, status = [], [], []
    for _ in range(iters):
        movers.append(((sp.env.state[4] >> 48) & 1).cpu().numpy())
        sp.step(restart=False)
        values.append(sp.resign_value.cpu().numpy().copy())
        status.append((sp.env.state[4] >> 56).cpu().numpy())
        if sp.running() == 0:
            break
    return sp, np.array(movers), np.array(values), np.array(status)


def slot_values(movers, values, s):
    return [(int(movers[k, s]), float(values[k, s]), k) for k in range(len(values)) if not math.isnan(values[k, s])]


def test_resigned_games_are_prefixes_of_track_only_games(model, calib):
    n, iters, P = 160, 260, 2
    kw = dict(num_itr=12, seed=41, resign_plies=P, resign_probe=0.0)
    a, ma, va, sa = logged_run(model, n, iters, resign_threshold=-1.0, **kw)
    b, mb, vb, sb = logged_run(model, n, iters, resign_threshold=calib, **kw)
    R = min(len(sa), len(sb))
    rs_a, vis_a, fl_a = (a.rec_state.view(iters, n, 5), a.rec_visits.view(iters, n, 294), a.rec_flag.view(iters, n))
    rs_b, vis_b, fl_b = (b.rec_state.view(iters, n, 5), b.rec_visits.view(iters, n, 294), b.rec_flag.view(iters, n))
    resigned = 0
    for s in range(n):
        vals = slot_values(ma, va, s)
        at, who, _ = resign_ref.track_game([(p, r) for p, r, _ in vals], calib, P, probe=False)
        if at is None:
            assert torch.equal(rs_a[:, s], rs_b[:, s]) and torch.equal(vis_a[:, s], vis_b[:, s]) and torch.equal(fl_a[:, s], fl_b[:, s])
            assert torch.equal(a.env.state[:, s], b.env.state[:, s])
            continue
        resigned += 1
        k = vals[at][2]                                  # the iteration whose search resigned
        assert sb[k, s] == (8 if who == 0 else 7) and (k == 0 or sb[k - 1, s] == 0) and np.all(sb[k:R, s] == sb[k, s])
        assert np.allclose(vb[:k + 1, s], va[:k + 1, s], equal_nan=True)
        assert torch.equal(rs_a[:k, s], rs_b[:k, s]) and torch.equal(vis_a[:k, s], vis_b[:k, s])
        movers = ((rs_b[:k, s, 4] >> 48) & 1).cpu().numpy()
        flags = (fl_b[:k, s] & 0xF).cpu().numpy()
        recorded = (fl_a[:k, s] & 0xF).cpu().numpy() != 0
        assert np.array_equal(flags[recorded], np.where(movers[recorded] == who, 3, 2))   # a win for the side that did not resign
        assert not np.any(flags[~recorded]) and not bool((fl_b[k:, s] & 0xF).any())
    assert resigned > 5 and b.stats()["resigned_games"] == resigned


def test_probe_games(model, calib):
    # every game a probe: the run is the track-only run
    kw = dict(n_slots=128, num_itr=12, max_iters=400, seed=17, resign_plies=2)
    a = drain_result(sp_of(model, resign_threshold=-1.0, **kw), 200)
    b = drain_result(sp_of(model, resign_threshold=calib, resign_probe=1.0, **kw), 200)
    assert {k: a[0][k] for k in BASE_KEYS} == {k: b[0][k] for k in BASE_KEYS} and torch.equal(a[2], b[2])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k
    assert b[0]["resigned_games"] == 0 and b[0]["probe_games"] == b[0]["p1_wins"] + b[0]["p2_wins"]
    # one game in ten a probe, over 4,096 games: share, would-resigns, false positives and samples as the host rule says
    n, iters, P, f = 4096, 400, 2, 0.1
    sp, mv, val, status = logged_run(model, n, iters, num_itr=6, seed=29, resign_threshold=calib, resign_plies=P, resign_probe=f)
    probe = (sp.resign_state[:, 1] & 1).cpu().numpy().astype(bool)
    assert np.all(sp.serial.cpu().numpy() == 0)
    sd = math.sqrt(n * f * (1 - f))
    assert abs(probe.sum() - n * f) <= 3.29 * sd, probe.sum()
    final = status[-1]
    would = fps = resigned = 0
    samples = []
    for s in range(n):
        vals = slot_values(mv, val, s)
        at, who, wmin = resign_ref.track_game([(p, r) for p, r, _ in vals], calib, P, probe=bool(probe[s]))
        if not probe[s]:
            resigned += at is not None
            assert (final[s] in (7, 8)) == (at is not None)
            continue
        if final[s] in (1, 2):
            would += who is not None
            fps += who is not None and who == final[s] - 1
            samples.append((int(np.argmax(status[:, s] != 0)), s, wmin[final[s] - 1]))
    st = sp.stats()
    assert st["resigned_games"] == resigned > 0
    assert st["probe_games"] == sum(1 for s in range(n) if probe[s] and final[s] in (1, 2))
    assert st["probe_would_resign"] == would and st["probe_false_positives"] == fps
    got = sp.resign_samples()
    assert st["resign_samples_written"] == len(samples) == len(got) and st["resign_samples_dropped"] == 0
    assert np.array_equal(got, np.array([x[2] for x in sorted(samples)]))


def test_compaction_changes_nothing_with_resignation(model, calib):
    def run(compact):
        sp = sp_of(model, n_slots=320, seed=9, num_itr=10, max_iters=400, resign_threshold=calib, resign_plies=1, resign_probe=0.1)
        st = sp.play_games(400, compact=compact, compact_min=24)
        t = sp.collect()
        key = np.vstack([t["state"].cpu().numpy(), t["v_y"].cpu().numpy()[None].astype(np.int64),
                         (t["pi_y"].double() * torch.arange(1, 295, device=t["pi_y"].device)).sum(1).mul(1e6).round().long().cpu().numpy()[None]])
        order = np.lexsort(key)
        return st, t["board_x"].cpu().numpy()[order], t["pi_y"].cpu().numpy()[order], t["v_y"].cpu().numpy()[order], sp.resign_samples(), sp.n
    a, b = run(False), run(True)
    assert b[0]["compactions"] >= 1 and a[0]["compactions"] == 0 and b[5] < a[5]
    assert {k: v for k, v in a[0].items() if k != "compactions"} == {k: v for k, v in b[0].items() if k != "compactions"}
    assert a[0]["resigned_games"] > 0 and a[1].shape[0] == a[0]["records"] > 0
    for x, y in zip(a[1:5], b[1:5]):
        assert np.array_equal(x, y)


def test_two_nets_with_twin_nets_equal_one_net(model, calib):
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    eng2 = Engine(0)
    try:
        m2 = ResidualCNN(engine=eng2).load_weights(WEIGHTS)
        kw = dict(n_slots=96, num_itr=12, max_iters=120, seed=13, log_moves=True, resign_threshold=calib, resign_plies=1, resign_probe=0.1)
        a = sp_of(model, **kw)
        a.run(iters=120)
        b = sp_of(model, opponent=m2, **kw)
        b.run(iters=120)
        assert torch.equal(a.move_log, b.move_log) and torch.equal(a.rec_visits, b.rec_visits) and torch.equal(a.rec_flag, b.rec_flag)
        assert torch.equal(a.env.state, b.env.state) and torch.equal(a.resign_state, b.resign_state)
        assert a.stats() == b.stats() and a.stats()["resigned_games"] > 0
        assert np.array_equal(a.resign_samples(), b.resign_samples())
    finally:
        eng2.close()


def test_evolve_calibrates_the_threshold(tmp_path):
    from chinesecheckersagent_b200.train import evolve
    logs = []
    cur, best, it = evolve(WEIGHTS, None, 0, None, max_iterations=2, num_self_play=24, data_dir=str(tmp_path / "data"),
                           weights_dir=str(tmp_path / "weights"), seed=5, epochs=1, log=logs.append, n_slots=24, num_itr=12,
                           max_iters=400, resign_fp=0.05)
    assert it == 2 and os.path.exists(cur)
    used = [m for m in logs if "resign threshold" in m]
    assert len(used) == 2 and "iteration 0: self-play resign threshold -1.000000" in used[0]
    assert "resigned_games" in " ".join(m for m in logs if "self-play with" in m)


def test_arguments_are_checked(model):
    for bad in (dict(resign_threshold=1.5), dict(resign_threshold=-2.0), dict(resign_threshold=float("nan")),
                dict(resign_threshold=0.0, resign_plies=0), dict(resign_threshold=0.0, resign_plies=9),
                dict(resign_threshold=0.0, resign_probe=1.5), dict(resign_threshold=0.0, resign_samples=-1)):
        with pytest.raises(ValueError):
            sp_of(model, n_slots=8, **bad)
