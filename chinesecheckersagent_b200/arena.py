"""Arena / evaluation games on the device (§8f f2): the reference's ai_vs_ai.agent_match (ai_vs_ai.py:28-52),
ai_vs_greedy.agent_greedy_match (ai_vs_greedy.py:26-59) and train.evaluate (train.py:150-187) with every game of a
match played at once: `Game.start` semantics (game.py:58-100) per ply for all games, the AiPlayer's
MCTS (player.py:136-166: search on the unexpanded root, 175 simulations, move sampled from N^(1/tau)) batched over
the games whose mover uses that model.

Two models = two `ResidualCNN`s, each living in its own `Engine` (own weights, own tree pools) on the same GPU;
the game states are plain device tensors both engines read and write."""
import torch

from .config import (C_PUCT, DEFAULT_SEED, DET_TREE_TAU, EVAL_GAMES, MCTS_SIMULATIONS, PLAYER_ONE, PLAYER_TWO,
                     PROGRESS_MOVE_LIMIT, ST_OVERFLOW, ST_RUNNING, TOTAL_MOVES_TILL_TAU0)
from .engine import BatchedEnv, BatchedMCTS, _p

GREEDY = "greedy"


class BatchedArena:
    """n games, player 1 = `p1`, player 2 = `p2`; each is a loaded ResidualCNN or the string "greedy"."""

    def __init__(self, p1, p2, n, seed=DEFAULT_SEED, game_id0=0, tree_tau=DET_TREE_TAU, enforce_move_limit=False,
                 num_itr=MCTS_SIMULATIONS, cpuct=C_PUCT, random_ties=True, leaves_per_round=1, reuse_tree=False, gumbel=False):
        """random_ties: PUCT ties drawn uniformly like the reference's random.choice (MCTS.py:65-72), keyed per game — without
        it (first maximal edge) every game of a match between two deterministic players at tau = 0.01 is the same game.
        leaves_per_round: leaves per tree per search round (BatchedMCTS), one int for both sides or a (player 1, player 2)
        pair, so that a match can pit a leaf-parallel search against the one-leaf search.
        reuse_tree: tree reuse (BatchedMCTS reuse_tree), one bool for both sides or a (player 1, player 2) pair.  A side whose
        engine searched only its own plies continues its tree at depth 2 (its move and the reply).  Two sides sharing one
        engine share its tree pool, so each continues the opponent's last tree at depth 1; for an A/B test of reuse with one
        net, load the net into two engines.
        gumbel: Gumbel search (BatchedMCTS gumbel=True, defaults of its gumbel_* parameters, draws keyed by the seed and the game),
        one bool for both sides or a pair; a Gumbel side plays its search's action.  num_itr may be a pair as well, so that
        searches of different sizes can meet."""
        models = [p for p in (p1, p2) if p is not GREEDY and p != GREEDY]
        if not models:
            raise ValueError("at least one side must be a model (greedy-vs-greedy is BatchedEnv.play_greedy)")
        if len(models) == 2 and models[0] is not models[1] and models[0].eng is models[1].eng:
            raise ValueError("two different models need two Engines (one set of net weights per ccx handle)")
        self.players = {PLAYER_ONE: p1, PLAYER_TWO: p2}
        self.n, self.seed, self.uid0 = int(n), int(seed), int(game_id0)
        self.tau = float(tree_tau)
        self.move_limit = PROGRESS_MOVE_LIMIT if enforce_move_limit else 0
        self.eng = models[0].eng                                   # owns the game states and the bookkeeping kernel
        self.env = BatchedEnv(self.n, engine=self.eng, seed=seed, game_id0=game_id0)
        self.counters = self.eng.zeros((4,), torch.int64)
        leaves = tuple(leaves_per_round) if isinstance(leaves_per_round, (tuple, list)) else (leaves_per_round,) * 2
        reuse = tuple(reuse_tree) if isinstance(reuse_tree, (tuple, list)) else (reuse_tree,) * 2
        gum = tuple(gumbel) if isinstance(gumbel, (tuple, list)) else (gumbel,) * 2
        itr = tuple(num_itr) if isinstance(num_itr, (tuple, list)) else (num_itr,) * 2
        self.mcts = {side: BatchedMCTS(p.eng, cpuct=cpuct, num_itr=I, random_ties=random_ties, tie_seed=seed ^ 0xA7E4A,
                                       tie_uid0=game_id0, leaves_per_round=L, reuse_tree=R, gumbel=G, gumbel_seed=seed ^ 0x6B3E1)
                     for side, p, L, R, G, I in ((PLAYER_ONE, p1, leaves[0], reuse[0], gum[0], itr[0]),
                                                 (PLAYER_TWO, p2, leaves[1], reuse[1], gum[1], itr[1]))
                     if p is not GREEDY and p != GREEDY}
        self.plies = 0

    def step(self):
        """one ply of every running game (all games of a match have the same side to move)"""
        side = PLAYER_ONE if self.plies % 2 == 0 else PLAYER_TWO
        mover = self.players[side]
        st = self.env.state
        if mover == GREEDY:
            self.eng.call("ccx_game_advance", self.n, _p(st), None, None, self.seed, self.uid0, self.tau, TOTAL_MOVES_TILL_TAU0,
                          self.move_limit, _p(self.counters))
        else:
            # (both engines launch on torch's current stream, so their kernels are ordered without extra synchronisation)
            res = self.mcts[side].search_net(st, pre_expand=False, min_ply_status=True)
            if "action" in res:                                     # Gumbel: the action as one-hot visits, which the sampler plays
                act = res["action"].long()
                res["visits"].zero_().scatter_(1, act.clamp(min=0).unsqueeze(1), (act >= 0).int().unsqueeze(1))
            self.eng.call("ccx_game_advance", self.n, _p(st), _p(res["visits"]), _p(res["n_nodes"]), self.seed, self.uid0, self.tau,
                          TOTAL_MOVES_TILL_TAU0, self.move_limit, _p(self.counters))
        self.plies += 1

    def running(self):
        return int(((self.env.state[4] >> 56) == ST_RUNNING).sum().item())

    def play(self, max_plies=1000, poll_every=4):
        while self.plies < max_plies:
            self.step()
            if self.plies % poll_every == 0 and self.running() == 0:
                break
        c = self.counters.cpu().tolist()
        overflowed = int(((self.env.state[4] >> 56) == ST_OVERFLOW).sum().item())     # a search ran out of edge pool: not a draw
        return dict(plies=c[0], p1_wins=c[1], p2_wins=c[2], stopped=c[3], overflowed=overflowed, unfinished=self.running(),
                    games=self.n)


def _load(model_or_path, engine=None):
    from .model import ResidualCNN
    if isinstance(model_or_path, ResidualCNN) or model_or_path == GREEDY:
        return model_or_path
    from .engine import Engine
    return ResidualCNN(engine=engine or Engine()).load_weights(model_or_path)


def agent_match(model1_path, model2_path, num_games, verbose=False, tree_tau=DET_TREE_TAU, enforce_move_limit=False, seed=DEFAULT_SEED):
    """ai_vs_ai.py:28-52 — model1 plays player 1 in every game; returns the winner's path by the 55 % rule, else None."""
    m1, m2 = _load(model1_path), _load(model2_path)
    res = BatchedArena(m1, m2, num_games, seed=seed, tree_tau=tree_tau, enforce_move_limit=enforce_move_limit).play()
    if verbose:
        print('Agent "{}" wins {} matches'.format(model1_path, res["p1_wins"]))
        print('Agent "{}" wins {} matches'.format(model2_path, res["p2_wins"]))
    if res["p1_wins"] > int(0.55 * num_games):
        return model1_path
    if res["p2_wins"] > int(0.55 * num_games):
        return model2_path
    return None


def agent_greedy_match(model_path, num_games, verbose=False, tree_tau=DET_TREE_TAU, seed=DEFAULT_SEED):
    """ai_vs_greedy.py:26-59 — sides alternate game by game (the model is player 1 in games 0, 2, ...)."""
    m = _load(model_path)
    n1 = (num_games + 1) // 2
    a = BatchedArena(m, GREEDY, n1, seed=seed, tree_tau=tree_tau).play()
    b = BatchedArena(GREEDY, m, num_games - n1, seed=seed, game_id0=n1, tree_tau=tree_tau).play() if num_games > n1 else dict(p1_wins=0, p2_wins=0)
    ai, greedy = a["p1_wins"] + b["p2_wins"], a["p2_wins"] + b["p1_wins"]
    if verbose:
        print('Agent wins {} games and Greedy wins {} games with total games {}'.format(ai, greedy, num_games))
    return model_path if ai > greedy else (GREEDY if greedy > ai else None)


def evaluate(best_model, cur_model, num_games=EVAL_GAMES, seed=DEFAULT_SEED):
    """train.evaluate (train.py:150-187): colours alternate, move limit enforced; returns (cur wins, best wins, draws)."""
    best, cur = _load(best_model), _load(cur_model)
    n_even = (num_games + 1) // 2                                   # games 0, 2, ...: best is player 1
    a = BatchedArena(best, cur, n_even, seed=seed, enforce_move_limit=True).play()
    b = (BatchedArena(cur, best, num_games - n_even, seed=seed, game_id0=n_even, enforce_move_limit=True).play()
         if num_games > n_even else dict(p1_wins=0, p2_wins=0))
    cur_wins, best_wins = a["p2_wins"] + b["p1_wins"], a["p1_wins"] + b["p2_wins"]
    return cur_wins, best_wins, num_games - cur_wins - best_wins
