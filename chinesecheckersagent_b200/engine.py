"""Batched env engine: torch owns the device memory, libccx.so's sm_100a kernels do the work.

`BatchedEnv` is the batched counterpart of the reference's `Board` (board.py): one SoA state tensor of
shape (8, n) int64 on the GPU holds n independent games (layout: include/ccx.h)."""
import ctypes

import numpy as np
import torch

from . import _lib
from .config import (DEFAULT_SEED, DTYPE_BF16, DTYPE_F32, DTYPE_U8, RESET_RANDOMISED, RESET_START,
                     STATE_WORDS, TRACE_WORDS)

_TORCH_DTYPE = {DTYPE_U8: torch.uint8, DTYPE_BF16: torch.bfloat16, DTYPE_F32: torch.float32}


class Engine:
    """One ccx handle bound to one CUDA device; kernels run on torch's current stream."""

    def __init__(self, device=None):
        """device: CUDA ordinal / torch.device; None = torch's current CUDA device (rank r of a multi-GPU job: device r)"""
        if not torch.cuda.is_available():
            raise _lib.CcxError("no CUDA device: the ccx engine has no CPU path")
        self.L = _lib.load()
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        h = ctypes.c_void_p()
        _lib.check(self.L, None, self.L.ccx_create(self.device.index, ctypes.byref(h)))
        self.h = h
        self._bind_stream()

    def _bind_stream(self):
        s = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.L, self.h, self.L.ccx_set_stream(self.h, ctypes.c_void_p(s)))

    def close(self):
        if getattr(self, "h", None):
            self.L.ccx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(self.L.ccx_launch_count(self.h))

    def call(self, name, *args):
        self._bind_stream()
        _lib.check(self.L, self.h, getattr(self.L, name)(self.h, *args))

    # -- tensor helpers -------------------------------------------------------------------------
    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def zeros(self, shape, dtype):
        return torch.zeros(shape, dtype=dtype, device=self.device)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class BatchedEnv:
    """n games in SoA form on the GPU.  Mirrors Board's methods for a batch (board.py:9-288)."""

    def __init__(self, n, engine=None, device=None, seed=DEFAULT_SEED, game_id0=0, randomised=False, state=None):
        self.eng = engine or Engine(device)
        self.n = int(n)
        self.seed = int(seed)
        self.game_id0 = int(game_id0)
        self.step_index = 0
        self.state = self.eng.empty((STATE_WORDS, self.n), torch.int64)
        self.wins = self.eng.zeros((2,), torch.int64)
        if state is not None:
            self.load_state(state)
        else:
            self.reset(randomised)

    # Board() / Board(randomised=True)
    def reset(self, randomised=False):
        self.eng.call("ccx_reset", self.n, _p(self.state), RESET_RANDOMISED if randomised else RESET_START,
                      self.seed, self.game_id0)
        self.step_index = 0

    def load_state(self, st):
        """st: numpy uint64 / torch int64 array of shape (8, n) in the include/ccx.h layout."""
        if isinstance(st, np.ndarray):
            st = torch.from_numpy(np.ascontiguousarray(st).view(np.int64))
        self.state.copy_(st.to(self.eng.device, non_blocking=False))

    def numpy_state(self):
        return self.state.cpu().numpy().view(np.uint64)

    # Board.get_valid_moves for the side to move -> (6, n) destination bitboards
    def movegen(self, out=None):
        out = out if out is not None else self.eng.empty((6, self.n), torch.int64)
        self.eng.call("ccx_movegen", self.n, _p(self.state), _p(out))
        return out

    # Board.place -> winner (n,) uint8
    def apply(self, frm, to, winner=None):
        winner = winner if winner is not None else self.eng.empty((self.n,), torch.uint8)
        self.eng.call("ccx_apply", self.n, _p(self.state), _p(frm), _p(to), _p(winner))
        return winner

    # check_win, player_progress(1|2), player_forward_distance(1|2) -> (n, 5) int16
    def info(self):
        out = self.eng.empty((self.n, 5), torch.int16)
        self.eng.call("ccx_info", self.n, _p(self.state), _p(out))
        return out

    def step_random(self, plies, trace_games=0):
        """`plies` fused random-legal env steps per game (selfplay.py:83-104 move choice)."""
        trace = None
        if trace_games:
            trace = self.eng.zeros((plies, trace_games, TRACE_WORDS), torch.int64)
        self.eng.call("ccx_step_random", self.n, _p(self.state), self.game_id0, self.seed, self.step_index,
                      int(plies), _p(self.wins), _p(trace), int(trace_games))
        self.step_index += int(plies)
        return trace

    def greedy_candidates(self):
        out = self.eng.empty((6, self.n), torch.int64)
        self.eng.call("ccx_greedy_candidates", self.n, _p(self.state), _p(out))
        return out

    def play_greedy(self, max_plies=100000, counters=None):
        """Game('greedy','greedy').start() for every running game (game.py:58-100)."""
        counters = counters if counters is not None else self.eng.zeros((4,), torch.int64)
        self.eng.call("ccx_play_greedy", self.n, _p(self.state), self.game_id0, self.seed, int(max_plies), _p(counters))
        return counters

    def encode(self, dtype=DTYPE_BF16, out=None):
        """utils.to_model_input for every game -> (n, 7, 7, 7) channels-last."""
        out = out if out is not None else self.eng.empty((self.n, 7, 7, 7), _TORCH_DTYPE[dtype])
        self.eng.call("ccx_encode", self.n, _p(self.state), _p(out), dtype)
        return out


class HostEnv:
    """The reference-facing path with HOST buffers: numpy in, numpy out, H2D/D2H inside each call."""

    def __init__(self, engine=None, device=None):
        self.eng = engine or Engine(device)

    @staticmethod
    def _np(a):
        return ctypes.c_void_p(a.ctypes.data)

    def movegen(self, st):
        n = st.shape[1]
        masks = np.empty((6, n), dtype=np.uint64)
        self.eng.call("ccx_movegen_host", n, self._np(st), self._np(masks))
        return masks

    def apply(self, st, frm, to):
        n = st.shape[1]
        winner = np.empty(n, dtype=np.uint8)
        self.eng.call("ccx_apply_host", n, self._np(st), self._np(frm), self._np(to), self._np(winner))
        return winner

    def step_random(self, st, plies, seed=DEFAULT_SEED, step0=0, game_id0=0, wins=None):
        wins = wins if wins is not None else np.zeros(2, dtype=np.uint64)
        self.eng.call("ccx_step_random_host", st.shape[1], self._np(st), game_id0, seed, step0, int(plies), self._np(wins))
        return wins

    def encode(self, st, dtype=DTYPE_U8):
        n = st.shape[1]
        npdt = {DTYPE_U8: np.uint8, DTYPE_BF16: np.uint16, DTYPE_F32: np.float32}[dtype]
        out = np.empty((n, 7, 7, 7), dtype=npdt)
        self.eng.call("ccx_encode_host", n, self._np(st), self._np(out), dtype)
        return out


EVAL_UNIFORM, EVAL_HASH = 0, 1
MAX_LEAVES = 16                 # include/ccx.h CCX_MAX_LEAVES
REUSE_CARRY = 3                 # default carry of tree reuse (DESIGN.md §3, tree reuse)


class BatchedMCTS:
    """Batched counterpart of MCTS.MCTS (MCTS.py:40-153): one tree per root state, all trees advanced one
    simulation at a time; returns visit-count policies."""

    def __init__(self, engine, cpuct=3.5, num_itr=175, tree_tau=1.0, edges_per_tree=0, random_ties=False, tie_seed=DEFAULT_SEED,
                 tie_uid0=0, leaves_per_round=1, reuse_tree=False, reuse_carry=REUSE_CARRY, gumbel=False, gumbel_considered=16,
                 gumbel_scale=1.0, gumbel_c_visit=50.0, gumbel_c_scale=0.1, gumbel_seed=DEFAULT_SEED):
        """random_ties=False: PUCT ties go to the first maximal edge (bit-exact parity mode); True: the reference's rule
        (MCTS.py:65-72: uniform among the epsilon-tie list), drawn with Philox keyed by (tie_seed, tie_uid0 + tree index).
        leaves_per_round=L > 1 (search_with, search_net): each round selects up to L leaves per tree under virtual loss and
        evaluates them in one batch of n*L positions (include/ccx.h, ccx_mcts_select_leaves): about 1 + (num_itr - 1) / L
        rounds per search instead of num_itr; 1 = the reference's one simulation at a time.
        reuse_tree=True (search_with, search_net): each search starts, tree by tree, from the subtree the previous search on
        this engine grew below the new root (matched by state at depth 1 or 2; include/ccx.h, ccx_mcts_begin_reuse), when it
        holds no more than reuse_carry times one search's nodes, edges and visits; otherwise fresh.  The results then carry
        `reused` (n,) int32: 1 / 2 = depth of the match, 0 = fresh, -2 = inactive.  The evaluator must stay the same from
        search to search (loading weights into the engine starts every tree fresh); pass `prev` to a search after reordering
        or dropping roots: prev[i] = index of root i in the previous search, -1 = none.
        gumbel=True (search_with, search_net): Gumbel search (include/ccx.h, ccx_mcts_set_gumbel) instead of PUCT: the root's
        moves are Gumbel-top-k sampled (gumbel_considered = m, gumbel_scale = the draws' scale, 0 = deterministic, gumbel_seed keys
        them with tie_uid0 + tree index) and visited by sequential halving, interior nodes take argmax pi' - N / (1 + sum N);
        the results add `action` (n,) int32, the move to play, and `pi` is the improved policy softmax(logit + sigma(Q)).
        num_itr counts the rounds as for PUCT (pre_expand adds the root's expansion), tree_tau and the tie rule do not apply.
        Not with leaves_per_round > 1, reuse_tree or search().  The engine is in the mode only during this object's searches."""
        self.eng = engine
        self.cpuct, self.num_itr, self.tree_tau, self.edges_per_tree = float(cpuct), int(num_itr), float(tree_tau), int(edges_per_tree)
        self.random_ties, self.tie_seed, self.tie_uid0 = bool(random_ties), int(tie_seed), int(tie_uid0)
        self.leaves = int(leaves_per_round)
        if not 1 <= self.leaves <= MAX_LEAVES:
            raise ValueError("leaves_per_round must be in 1..%d" % MAX_LEAVES)
        self.reuse_tree, self.reuse_carry = bool(reuse_tree), int(reuse_carry)
        if self.reuse_carry < 0:
            raise ValueError("reuse_carry must be >= 0")
        self.gumbel = bool(gumbel)
        self.gumbel_params = (int(gumbel_considered), float(gumbel_scale), float(gumbel_c_visit), float(gumbel_c_scale),
                              int(gumbel_seed) & 0xFFFFFFFFFFFFFFFF)
        if self.gumbel:
            if self.leaves != 1 or self.reuse_tree:
                raise ValueError("the Gumbel search runs one leaf per round on fresh trees: no leaves_per_round > 1, no reuse_tree")
            if self.gumbel_params[0] < 1 or min(self.gumbel_params[1:4]) < 0:
                raise ValueError("gumbel_considered must be >= 1 and the Gumbel scales >= 0")

    def _gumbel_search(self, roots, pre_expand, root_noise, prev, min_ply_status, run):
        """one Gumbel search: the mode is on only between set and finalize, so other users of the engine are unaffected"""
        if root_noise is not None or prev is not None:
            raise ValueError("the Gumbel search takes no root_noise (its draws are the exploration) and no prev (no tree reuse)")
        n, e = roots.shape[1], self.eng
        rounds = self.num_itr + (1 if pre_expand else 0)
        self._tie_rule()                                 # tie_uid0 keys the Gumbel draws
        e.call("ccx_mcts_set_gumbel", 1, *self.gumbel_params)
        try:
            e.call("ccx_mcts_begin", n, _p(roots), rounds, self.edges_per_tree, 0 if min_ply_status else -1, -1)
            run(n, rounds)
            visits, pi, q, nodes = self._outputs(n)
            action = e.empty((n,), torch.int32)
            e.call("ccx_mcts_finalize_gumbel", n, _p(visits), _p(pi), _p(q), _p(action), _p(nodes))
        finally:
            e.call("ccx_mcts_set_gumbel", 0, 1, 0.0, 0.0, 0.0, 0)
        out = self._result(visits, pi, q, nodes, None)
        out["action"] = action
        return out

    def _tie_rule(self):
        self.eng.call("ccx_mcts_set_tiebreak", 1 if self.random_ties else 0, self.tie_seed, self.tie_uid0)

    def _begin(self, roots, min_ply, root_noise, stride, prev):
        """begin a search (ccx_mcts_begin, or ccx_mcts_begin_reuse with the root noise for carried roots); returns `reused`"""
        n = roots.shape[1]
        if not self.reuse_tree:
            if prev is not None:
                raise ValueError("prev needs reuse_tree=True")
            self.eng.call("ccx_mcts_begin", n, _p(roots), self.num_itr + 1, self.edges_per_tree, min_ply, -1)
            return None
        if prev is not None and (prev.dtype != torch.int64 or tuple(prev.shape) != (n,) or not prev.is_contiguous()
                                 or prev.device != self.eng.device):
            raise ValueError("prev must be a contiguous int64 tensor of shape (n,) on the engine's device")
        reused = self.eng.empty((n,), torch.int32)
        self.eng.call("ccx_mcts_begin_reuse", n, _p(roots), self.num_itr + 1, self.edges_per_tree, min_ply, -1, self.reuse_carry,
                      _p(prev), _p(root_noise), stride, 0, _p(reused))
        return reused

    def _outputs(self, n, want_q=True):
        e = self.eng
        return (e.empty((n, 294), torch.int32), e.empty((n, 294), torch.float64),
                e.empty((n, 294), torch.float64) if want_q else None, e.empty((n,), torch.int32))

    def search(self, roots, evaluator=EVAL_UNIFORM, pre_expand=False, root_noise=None):
        """In-kernel evaluator (uniform stub / hash test evaluator).  roots: (8, n) int64 device tensor.
        Returns dict(visits, pi, q, n_nodes)."""
        if self.leaves != 1:
            raise ValueError("the in-kernel evaluators search one leaf per round: use search_with for leaves_per_round > 1")
        if self.gumbel:
            raise ValueError("the in-kernel evaluators search with PUCT: use search_with for the Gumbel search")
        n = roots.shape[1]
        visits, pi, q, nodes = self._outputs(n)
        stride = 0 if root_noise is None else root_noise.shape[1]
        self._tie_rule()
        self.eng.call("ccx_mcts_search", n, _p(roots), int(evaluator), self.num_itr, self.cpuct, self.tree_tau,
                      int(bool(pre_expand)), _p(root_noise), stride, self.edges_per_tree, _p(visits), _p(pi), _p(q), _p(nodes))
        return dict(visits=visits, pi=pi, q=q, n_nodes=nodes)

    def search_with(self, roots, evaluate, pre_expand=False, root_noise=None, prev=None, min_ply_status=False):
        """External evaluator: evaluate(leaf_state (5, n*L) int64) -> (p (n*L, 294) float64, v (n*L,) float64), L =
        leaves_per_round, slot i*L + k = leaf k of tree i.  One select / evaluate / expand+backup round per simulation
        (L = 1) or per up to L simulations of every tree.  prev, min_ply_status: as for search_net."""
        n = roots.shape[1]
        e = self.eng
        L = self.leaves
        leaf = e.empty((5, n * L), torch.int64)
        if self.gumbel:
            def rounds_with(n, rounds):
                for _ in range(rounds):
                    e.call("ccx_mcts_select", n, self.cpuct, _p(leaf))
                    p, v = evaluate(leaf)
                    e.call("ccx_mcts_expand_backup", n, _p(p), _p(v), None, 0, 0)
            return self._gumbel_search(roots, pre_expand, root_noise, prev, min_ply_status, rounds_with)
        stride = 0 if root_noise is None else root_noise.shape[1]
        self._tie_rule()
        reused = self._begin(roots, 0 if min_ply_status else -1, root_noise if pre_expand else None, stride, prev)
        rounds = self.num_itr + (1 if pre_expand else 0)
        if L > 1:
            # round 0 selects the unexpanded roots, later rounds up to L leaves of what is left
            e.call("ccx_mcts_leaf_budget", n, L, rounds)
            for r in range(1 + (rounds - 1 + L - 1) // L):
                e.call("ccx_mcts_select_leaves", n, L, self.cpuct, _p(leaf))
                p, v = evaluate(leaf)
                noise = root_noise if (pre_expand and r == 0) else None
                e.call("ccx_mcts_expand_backup_leaves", n, L, _p(p), _p(v), _p(noise), stride if noise is not None else 0, 0)
        else:
            for r in range(rounds):
                e.call("ccx_mcts_select", n, self.cpuct, _p(leaf))
                p, v = evaluate(leaf)
                noise = root_noise if (pre_expand and r == 0) else None
                e.call("ccx_mcts_expand_backup", n, _p(p), _p(v), _p(noise), stride if noise is not None else 0, 0)
        visits, pi, q, nodes = self._outputs(n)
        e.call("ccx_mcts_finalize", n, self.tree_tau, _p(visits), _p(pi), _p(q), _p(nodes))
        return self._result(visits, pi, q, nodes, reused)

    @staticmethod
    def _result(visits, pi, q, nodes, reused):
        out = dict(visits=visits, pi=pi, q=q, n_nodes=nodes)
        if reused is not None:
            out["reused"] = reused
        return out

    def search_net(self, roots, pre_expand=False, root_noise=None, min_ply_status=False, prev=None):
        """The library's own policy/value net as the evaluator (the weights loaded into this engine by
        model.ResidualCNN.load_weights), all rounds in one C call with the fused round kernels
        (ccx_mcts_run_net).  Same results as search_with(roots, model.evaluate_states, ...).
        prev (reuse_tree only): int64 (n,) device tensor, the previous search's index of root i (-1 = none)."""
        n = roots.shape[1]
        e = self.eng
        if self.gumbel:
            return self._gumbel_search(roots, pre_expand, root_noise, prev, min_ply_status,
                                       lambda n, rounds: e.call("ccx_mcts_run_net", n, rounds, self.cpuct, None, 0, 0))
        stride = 0 if root_noise is None else root_noise.shape[1]
        # min_ply_status: roots whose status is not RUNNING get an inactive tree (finished arena / self-play games)
        self._tie_rule()
        reused = self._begin(roots, 0 if min_ply_status else -1, root_noise if pre_expand else None, stride, prev)
        rounds = self.num_itr + (1 if pre_expand else 0)
        if self.leaves > 1:
            e.call("ccx_mcts_run_net_leaves", n, rounds, self.leaves, self.cpuct, _p(root_noise) if pre_expand else None, stride, 0)
        else:
            e.call("ccx_mcts_run_net", n, rounds, self.cpuct, _p(root_noise) if pre_expand else None, stride, 0)
        visits, pi, q, nodes = self._outputs(n)
        e.call("ccx_mcts_finalize", n, self.tree_tau, _p(visits), _p(pi), _p(q), _p(nodes))
        return self._result(visits, pi, q, nodes, reused)
