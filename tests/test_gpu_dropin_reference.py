"""The drop-in surface against the reference's own callers: the package's `Game` / `GreedyPlayer` / `AiPlayer` / `MCTS` /
`selfplay` (the modules a maintainer puts in front of the reference's flat modules) must reproduce what the UNMODIFIED
reference's game.py, player.py, MCTS.py and selfplay.py produced on the same inputs.  Those outputs are stored under
tests/golden/ (written by tests/golden/gen_golden*.py, which run the reference): greedy_games.npz (Game.start),
mcts_golden.npz (MCTS.search, AiPlayer path) and selfplay_golden.npz (selfplay.selfplay's ply log).  GPU only (the
facade has no CPU path)."""
import contextlib
import io
import os
import random

import numpy as np
import pytest

import oracle as orc
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

SEED = 0x5EED2026                                        # tests/golden/gen_golden.py


@pytest.fixture(scope="module")
def model():
    from chinesecheckersagent_b200.board import default_engine
    from chinesecheckersagent_b200.model import ResidualCNN
    return ResidualCNN(engine=default_engine()).load_weights(os.path.join(GOLDEN, "good_model_weights.npz"))


@pytest.fixture
def first_maximum_ties():
    """the stored searches ran the reference MCTS.py with random.choice pinned to the first candidate"""
    from chinesecheckersagent_b200.MCTS import MCTS
    old, MCTS.TIE_RULE = MCTS.TIE_RULE, "first"
    yield
    MCTS.TIE_RULE = old


def _rc(cell):
    return (int(cell) >> 3, int(cell) & 7)


def _board_and_player(words):
    from chinesecheckersagent_b200.board import Board
    return Board.from_packed(words), ((int(words[4]) >> 48) & 1) + 1


def test_reference_game_start_plays_greedy_games_on_the_facade_board():
    """game.py:58-100 + player.py:67-129: Game('greedy', 'greedy').start() with both GreedyPlayers picking among
    filtered_best_moves by the Philox rule of tests/golden/gen_golden.py; winner, ply count and final position of every
    game equal the reference's (greedy_games.npz)."""
    from chinesecheckersagent_b200 import board_utils
    from chinesecheckersagent_b200.game import Game
    from chinesecheckersagent_b200.player import GreedyPlayer
    gold = np.load(os.path.join(GOLDEN, "greedy_games.npz"))
    assert int(gold["seed"]) == SEED

    class PhiloxGreedy(GreedyPlayer):
        def __init__(self, player_num, gid, plies):
            GreedyPlayer.__init__(self, player_num)
            self.gid, self.plies = gid, plies

        def decide_move(self, board, verbose=False, training=False, total_moves=None):
            keyed = []
            for s, e in GreedyPlayer.decide_move(self, board, training=True):
                frm, to = board_utils.human_coord_to_np_index(s), board_utils.human_coord_to_np_index(e)
                keyed.append((board.checkers_id[self.player_num][frm] * 64 + orc.cell(*to), frm, to))
            keyed.sort()
            r = orc.philox(SEED & 0xFFFFFFFF, SEED >> 32, total_moves, 1, self.gid & 0xFFFFFFFF, self.gid >> 32)
            self.plies[0] += 1
            return keyed[(int(r[0]) * len(keyed)) >> 32][1:]
    for gid in range(60):
        plies = [0]
        g = Game(p1_type='greedy', p2_type='greedy', verbose=False)
        g.player_one, g.player_two = PhiloxGreedy(1, gid, plies), PhiloxGreedy(2, gid, plies)
        g.cur_player, g.next_player = g.player_one, g.player_two
        with contextlib.redirect_stdout(io.StringIO()):
            w = g.start()
        assert (w if w else 3) == gold["status"][gid] and plies[0] == gold["plies"][gid], gid
        assert np.array_equal(g.board.packed_state(1)[:4], gold["final"][:4, gid]), gid


def test_reference_selfplay_function_runs_on_the_facade(monkeypatch):
    """selfplay.py:11-80: the package's selfplay() replays, move for move, the games the reference's selfplay() played with
    scripted move pickers (selfplay_golden.npz).  Which plies are random opening plies and which are searched, the tree_tau
    of every search, where the game ends, whether it is discarded, the reward and the history length must all agree."""
    import chinesecheckersagent_b200.MCTS as mcts_mod
    from chinesecheckersagent_b200.config import DET_TREE_TAU
    from chinesecheckersagent_b200.selfplay import selfplay
    gold = np.load(os.path.join(GOLDEN, "selfplay_golden.npz"))

    class Script:
        def __init__(self, log):
            self.log, self.k, self.played, self.start = log, 0, [], None

        def next_move(self):
            f, t = self.log[self.k][:2]                  # IndexError: the facade plays on where the reference stopped
            return _rc(f), _rc(t)

        def choice(self, seq):                           # the opening's two random.choice calls (start, then destination)
            f, t = self.next_move()
            if self.start is None:
                assert f in seq
                self.start = f
                return f
            assert t in seq
            self.start = None
            self.played.append((orc.cell(*f), orc.cell(*t), 0, 0))
            self.k += 1
            return t

    class ScriptedMCTS:
        """MCTS(root, model, num_itr, tree_tau) whose search plays the logged move"""
        script = None

        def __init__(self, root, model, cpuct=None, num_itr=None, tree_tau=None):
            self.root, self.tree_tau = root, tree_tau

        def expandAndBackUp(self, leafNode, breadcrumbs):
            f, t = self.script.next_move()
            assert t in self.root.state.get_valid_moves(self.root.currPlayer)[f]
            self.root.edges = [mcts_mod.Edge(self.root, None, 1.0, f, t)]

        def search(self):
            root, e = self.root, self.root.edges[0]
            cid = root.state.checkers_id[root.currPlayer][e.fromPos]
            root.pi[cid * 49 + e.toPos[0] * 7 + e.toPos[1]] = 1.0
            self.script.played.append((orc.cell(*e.fromPos), orc.cell(*e.toPos), 1, int(self.tree_tau == DET_TREE_TAU)))
            self.script.k += 1
            return root.pi, e

    monkeypatch.setattr(mcts_mod, "MCTS", ScriptedMCTS)
    for g in range(len(gold["n_plies"])):
        log = [tuple(int(x) for x in m) for m in gold["moves"][g, :gold["n_plies"][g]]]
        ScriptedMCTS.script = s = Script(log)
        with monkeypatch.context() as m:
            m.setattr(random, "choice", s.choice)
            np.random.seed(g)
            hist, reward = selfplay(object())
        assert s.played == log, g
        status = int(gold["status"][g])
        if status in (3, 4):                             # discarded: repetition / no progress
            assert hist is None and reward is None, g
        else:
            assert reward == (1 if status == 1 else -1) and len(hist) == gold["n_history"][g], g


def test_reference_ai_player_decides_a_move_on_the_facade(model, monkeypatch, first_maximum_ties):
    """player.py:133-166: AiPlayer(tree_tau=0.01).decide_move -> MCTS(node, model, tree_tau).search() on an unexpanded root.
    With the reference's hash test evaluator (restated below) the root visit counts and pi equal the reference MCTS.py's
    for that path (mcts_golden.npz configuration 4), and the move played is one the reference's pi supports."""
    import chinesecheckersagent_b200.player as player_mod
    from chinesecheckersagent_b200.game import Game
    gold = np.load(os.path.join(GOLDEN, "mcts_golden.npz"))
    evaluator, pre_expand, use_noise, tau, num_itr = gold["configs"][4]
    assert (evaluator, pre_expand, use_noise, tau, num_itr) == (1, 0, 0, 0.01, 175)
    trees, base = [], player_mod.MCTS

    class Recorded(base):
        def __init__(self, *a, **k):
            base.__init__(self, *a, **k)
            trees.append(self)
    monkeypatch.setattr(player_mod, "MCTS", Recorded)
    for r in (0, 9, 17, 31, 33, 38, 41, 46):             # opening, mid-game and late greedy roots
        board, player = _board_and_player(gold["roots"][:, r])
        np.random.seed(1)
        frm, to = player_mod.AiPlayer(player_num=player, model=HashModel(), tree_tau=0.01).decide_move(board)
        root = trees[-1].root
        for e in root.edges:
            idx = root.state.checkers_id[player][e.fromPos] * 49 + e.toPos[0] * 7 + e.toPos[1]
            assert e.stats['N'] == gold["visits4"][r, idx], r
        assert np.allclose(root.pi, gold["pi4"][r], rtol=1e-12, atol=1e-300), r
        assert gold["pi4"][r, root.state.checkers_id[player][frm] * 49 + to[0] * 7 + to[1]] > 0, r
    monkeypatch.undo()
    # and a full Game between the AiPlayer (the package's net) and the GreedyPlayer finishes
    with contextlib.redirect_stdout(io.StringIO()):
        np.random.seed(5); random.seed(5)
        winner = Game(p1_type='ai', p2_type='greedy', verbose=False, model1=model).start()
    assert winner in (1, 2, None)


class StubModel:
    version = 0

    def predict(self, x):
        assert x.shape == (7, 7, 7)
        return np.full(294, 1 / 294.), 0.0


def test_reference_mcts_py_over_the_facade_board_equals_the_device_tree(first_maximum_ties):
    """MCTS.py:49-137 with the uniform stub, random.choice pinned to the first candidate: the reference's visit counts, Q and
    pi (mcts_golden.npz configuration 0, 48 roots), the package's MCTS object over its Board (device tree) and the C oracle
    give one answer."""
    from chinesecheckersagent_b200.MCTS import MCTS, Node
    gold = np.load(os.path.join(GOLDEN, "mcts_golden.npz"))
    assert tuple(gold["configs"][0]) == (0, 0, 0, 1.0, 175)
    _, opi, _, _ = orc.mcts(gold["roots"], 175, 3.5, 1.0, 0, 0, nthreads=8)
    assert np.array_equal(opi, gold["pi0"])
    for r in range(gold["roots"].shape[1]):
        board, player = _board_and_player(gold["roots"][:, r])
        root = Node(board, player)
        np.random.seed(1)
        pi, _ = MCTS(root, StubModel(), num_itr=175).search()
        visits, q = np.zeros(294, np.uint32), np.zeros(294)
        for e in root.edges:
            idx = board.checkers_id[player][e.fromPos] * 49 + e.toPos[0] * 7 + e.toPos[1]
            visits[idx], q[idx] = e.stats['N'], e.stats['Q']
        assert np.array_equal(visits, gold["visits0"][r]) and np.array_equal(q, gold["q0"][r]), r
        assert visits.sum() == 174 and np.array_equal(pi, gold["pi0"][r]), r


# ---- the hash test evaluator of tests/golden/gen_golden_mcts.py (spec in oracle/ccx_oracle_mcts.c) --------------------
def _splitmix64(z):
    M64 = (1 << 64) - 1
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


_COEF = [_splitmix64(k + 1) for k in range(343)]


def _philox_vec(k0, k1, c0):
    """Philox4x32-10 over a vector of c0 counters with c1 = 7, c2 = c3 = 0; returns word 0."""
    c0 = c0.astype(np.uint64)
    c1 = np.full_like(c0, 7)
    c2 = np.zeros_like(c0)
    c3 = np.zeros_like(c0)
    m32 = np.uint64(0xFFFFFFFF)
    k0 = np.uint64(k0); k1 = np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m32, p1 & m32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m32, p0 & m32
        k0 = (k0 + np.uint64(0x9E3779B9)) & m32
        k1 = (k1 + np.uint64(0xBB67AE85)) & m32
    return c0


class HashModel:
    version = 0

    def predict(self, x):
        flat = np.asarray(x).astype(np.uint8).reshape(-1)
        h = 0
        for k in np.nonzero(flat)[0]:
            h = (h + _COEF[k] * int(flat[k])) & ((1 << 64) - 1)
        w = _philox_vec(h & 0xFFFFFFFF, h >> 32, np.arange(295))
        return w[:294].astype(np.float64) / 4294967296.0, float(w[294]) / 2147483648.0 - 1.0
