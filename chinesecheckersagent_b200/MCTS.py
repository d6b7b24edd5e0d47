"""Mirror of the reference's MCTS.py object surface (Node, Edge, MCTS) on top of the device tree pools.

`MCTS(root, model, cpuct, num_itr, tree_tau)`, `.expandAndBackUp(root, [])`, `.search() -> (pi, sampled_edge)`
behave like MCTS.py:40-153 for the way selfplay.py:114-133 and player.py:157-166 use them: the root's edges
are materialised as Edge objects (stats N/W/Q/P, fromPos/toPos, outNode) so callers can mix noise into
stats['P'] before search() and walk to `sampled_edge.outNode` afterwards.  The tree itself lives on the GPU.

`model` is any object with `.predict(x (7,7,7)) -> (p[294], v)` (MCTS.py:93).  When it is this package's
`ResidualCNN` living in the board's engine, all simulations of a search run inside libccx.so
(`ccx_mcts_run_net`, one tree: 3 kernels per simulation, replayed as a CUDA graph) — one C call per search instead
of 176 Python round trips; any other evaluator is called once per simulation like the reference does.

PUCT ties: `MCTS.TIE_RULE = "random"` (default) draws uniformly among the reference's epsilon-tie list
(MCTS.py:65-72), seeded from Python's `random` module like the reference's `random.choice`; `"first"` takes the
first maximal edge (the deterministic mode the oracle tests pin).

Leaves per round: `MCTS.LEAVES_PER_ROUND = L` (1..16, default 1 = the reference's one simulation at a time) selects up to L
leaves per round under virtual loss and evaluates them together (include/ccx.h, ccx_mcts_run_net_leaves): about
1 + (num_itr - 1) / L net rounds per search.  A foreign evaluator's `predict` is then called once per leaf slot of a round."""
import copy
import ctypes
import random

import numpy as np
import torch

from . import utils
from .config import BOARD_HEIGHT, BOARD_WIDTH, C_PUCT, MCTS_SIMULATIONS, NUM_CHECKERS, PLAYER_ONE, PLAYER_TWO, TREE_TAU
from .engine import _p

ROOT_STRIDE = 128
# byte offsets of the root snapshot inside one device buffer (one D2H copy per search): n_edges i32 | moves u16[S] | N u32[S] |
# W f64[S] | P f64[S]
_OFF_NE, _OFF_MV, _OFF_N, _OFF_W, _OFF_P = 0, 8, 8 + 2 * ROOT_STRIDE, 8 + 6 * ROOT_STRIDE, 8 + 14 * ROOT_STRIDE
_ROOT_BYTES = 8 + 22 * ROOT_STRIDE


class Node:
    def __init__(self, state, currPlayer):
        self.state = state
        self.currPlayer = currPlayer
        self.edges = []
        self.pi = np.zeros(NUM_CHECKERS * BOARD_WIDTH * BOARD_HEIGHT, dtype='float64')

    def isLeaf(self):
        return len(self.edges) == 0


class Edge:
    """MCTS.py:24-37.  `outNode` (the child position, MCTS.py:104-107) is built on first access: callers only ever walk to
    the sampled edge's child (selfplay.py:130-133), so the other ~25 `deepcopy + place` per search are never paid."""

    def __init__(self, inNode, outNode, prior, fromPos, toPos):
        self.inNode, self._out = inNode, outNode
        self.currPlayer = inNode.currPlayer
        self.fromPos, self.toPos = fromPos, toPos
        self.stats = {'N': 0, 'W': 0, 'Q': 0, 'P': prior}

    @property
    def outNode(self):
        if self._out is None:
            child = copy.deepcopy(self.inNode.state)
            child.place(self.inNode.currPlayer, self.fromPos, self.toPos)             # MCTS.py:104-105
            self._out = Node(child, PLAYER_ONE + PLAYER_TWO - self.inNode.currPlayer)
        return self._out

    @outNode.setter
    def outNode(self, node):
        self._out = node


class _DeviceScratch:
    """per-engine device buffers of the one-tree searches (root state in, root snapshot out)"""
    _by_engine = {}

    def __init__(self, eng):
        self.eng = eng
        self.root = eng.empty((8, 1), torch.int64)
        self.leaf = eng.empty((5, 1), torch.int64)
        self.snap = eng.empty((_ROOT_BYTES,), torch.uint8)
        self.snap_host = torch.empty((_ROOT_BYTES,), dtype=torch.uint8).pin_memory()
        self.priors = eng.empty((1, ROOT_STRIDE), torch.float64)
        self.priors_host = torch.zeros((1, ROOT_STRIDE), dtype=torch.float64).pin_memory()

    def leaves(self, L):
        """leaf-slot buffer (5, L) of the leaf-parallel rounds"""
        if getattr(self, "_leaves", None) is None or self._leaves.shape[1] != L:
            self._leaves = self.eng.empty((5, L), torch.int64)
        return self._leaves

    @classmethod
    def of(cls, eng):
        d = cls._by_engine.get(id(eng))
        if d is None or d.eng is not eng:
            d = cls._by_engine[id(eng)] = cls(eng)
        return d


class MCTS:
    TIE_RULE = "random"          # "first" = first maximal edge (deterministic; what the oracle tests use)
    LEAVES_PER_ROUND = 1         # > 1: leaves per tree per round under virtual loss (opt-in; changes the search)

    def __init__(self, root, model, cpuct=C_PUCT, num_itr=MCTS_SIMULATIONS, tree_tau=TREE_TAU):
        self.root, self.model, self.cpuct, self.num_itr, self.tree_tau = root, model, cpuct, num_itr, tree_tau
        self.leaves = int(self.LEAVES_PER_ROUND)
        self._eng = root.state._eng
        self._dev = _DeviceScratch.of(self._eng)
        self._begun = False
        # the library's own net in this engine: every simulation of a search stays inside libccx (ccx_mcts_run_net)
        self._native = (getattr(model, "fused_mcts", False) and getattr(model, "eng", None) is self._eng and
                        getattr(model, "loaded", False) and hasattr(model, "evaluate_states"))

    # -- device plumbing -----------------------------------------------------------------------------------
    def _begin(self):
        d, e = self._dev, self._eng
        st = torch.from_numpy(self.root.state._pack(self.root.currPlayer - 1).view(np.int64))
        d.root.copy_(st, non_blocking=False)
        rule = 1 if self.TIE_RULE == "random" else 0
        e.call("ccx_mcts_set_tiebreak", rule, random.getrandbits(63) if rule else 0, 0)
        e.call("ccx_mcts_begin", 1, _p(d.root), self.num_itr + 2, 0, -1, -1)
        if self._native:
            self.model.set_kernel(self.model.kernel)          # another model of this engine may have switched the net mode
            self.model.set_symmetry(self.model.symmetry, self.model.symmetry_seed)      # ... or its symmetry
        self._begun = True

    def _evaluate(self, leaf=None):
        """Model.predict on the selected leaf (MCTS.py:93) for an evaluator that is not the library's own net; leaf (5, k):
        one predict per slot."""
        leaf = self._dev.leaf if leaf is None else leaf
        if hasattr(self.model, "evaluate_states") and getattr(self.model, "eng", None) is self._eng:
            return self.model.evaluate_states(leaf)
        words = leaf.cpu().numpy().view(np.uint64)
        ps, vs = [], []
        for i in range(leaf.shape[1]):
            st = np.zeros((8, 1), dtype=np.uint64)
            st[:5, 0] = words[:, i]
            x = self.root.state._host().encode(st).astype(np.float64)
            p, v = self.model.predict(x)
            ps.append(np.asarray(p, dtype=np.float64).reshape(-1))
            vs.append(float(v))
        p = torch.from_numpy(np.ascontiguousarray(np.stack(ps))).to(self._eng.device)
        v = torch.tensor(vs, dtype=torch.float64, device=self._eng.device)
        return p, v

    def _simulate(self, count):
        """`count` x (moveToLeaf, expandAndBackUp) (MCTS.py:123-125); with LEAVES_PER_ROUND = L > 1 in rounds of up to L"""
        L = self.leaves
        if self._native:
            if L > 1:
                self._eng.call("ccx_mcts_run_net_leaves", 1, int(count), L, float(self.cpuct), None, 0, 0)
            else:
                self._eng.call("ccx_mcts_run_net", 1, int(count), float(self.cpuct), None, 0, 0)
            return
        if L > 1:
            if count <= 0:
                return
            leaf = self._dev.leaves(L)
            self._eng.call("ccx_mcts_leaf_budget", 1, L, int(count))
            for _ in range(1 + (int(count) - 1 + L - 1) // L):
                self._eng.call("ccx_mcts_select_leaves", 1, L, float(self.cpuct), _p(leaf))
                p, v = self._evaluate(leaf)
                self._eng.call("ccx_mcts_expand_backup_leaves", 1, L, _p(p), _p(v), None, 0, 0)
            return
        for _ in range(count):
            self._eng.call("ccx_mcts_select", 1, float(self.cpuct), _p(self._dev.leaf))
            p, v = self._evaluate()
            self._eng.call("ccx_mcts_expand_backup", 1, _p(p), _p(v), None, 0, 0)

    def _pull_root(self):
        d, e = self._dev, self._eng
        base = d.snap.data_ptr()
        at = lambda off: ctypes.c_void_p(base + off)
        e.call("ccx_mcts_get_root", 1, ROOT_STRIDE, at(_OFF_NE), at(_OFF_MV), at(_OFF_N), at(_OFF_W), at(_OFF_P))
        d.snap_host.copy_(d.snap, non_blocking=False)
        raw = d.snap_host.numpy()
        k = int(raw[_OFF_NE:_OFF_NE + 4].view(np.int32)[0])
        if k > ROOT_STRIDE:
            raise RuntimeError("root has %d edges, more than the snapshot stride %d" % (k, ROOT_STRIDE))
        return (k, raw[_OFF_MV:_OFF_MV + 2 * k].view(np.uint16).astype(np.int64), raw[_OFF_N:_OFF_N + 4 * k].view(np.uint32).copy(),
                raw[_OFF_W:_OFF_W + 8 * k].view(np.float64).copy(), raw[_OFF_P:_OFF_P + 8 * k].view(np.float64).copy())

    def _materialise_root_edges(self):
        root = self.root
        k, mv, N, W, P = self._pull_root()
        if not root.edges:
            for j in range(k):
                cid, to = int(mv[j]) >> 8, int(mv[j]) & 0xFF
                frm, dst = root.state.checkers_pos[root.currPlayer][cid], (to >> 3, to & 7)
                root.edges.append(Edge(root, None, float(P[j]), frm, dst))
        for j, e in enumerate(root.edges):
            e.stats['N'] = int(N[j]); e.stats['W'] = float(W[j])
            e.stats['Q'] = float(W[j]) / int(N[j]) if N[j] else 0
            e.stats['P'] = float(P[j])

    # -- MCTS.py API -----------------------------------------------------------------------------------------
    def expandAndBackUp(self, leafNode, breadcrumbs):
        """Only the root expansion of selfplay.py:117 is driven from Python; expansions inside search()
        happen on the device."""
        assert leafNode is self.root and not breadcrumbs and leafNode.isLeaf()
        self._begin()
        self._simulate(1)
        self._materialise_root_edges()

    def search(self):
        if not self._begun:
            self._begin()
        elif self.root.edges:
            # callers may have edited stats['P'] (Dirichlet noise, selfplay.py:121-124): push it to the device
            d = self._dev
            P = d.priors_host.numpy()
            P[0, :len(self.root.edges)] = [e.stats['P'] for e in self.root.edges]
            d.priors.copy_(d.priors_host, non_blocking=False)
            self._eng.call("ccx_mcts_set_root_priors", 1, ROOT_STRIDE, _p(d.priors))
        self._simulate(self.num_itr)                                            # MCTS.py:123-125
        self._materialise_root_edges()
        root = self.root
        for edge in root.edges:                                                 # MCTS.py:131-137
            cid = root.state.checkers_id[root.currPlayer][edge.fromPos]
            root.pi[utils.encode_checker_index(cid, edge.toPos)] = pow(edge.stats['N'], 1. / self.tree_tau)
        root.pi /= np.sum(root.pi)
        sampled_index = np.random.choice(np.arange(len(root.pi)), p=root.pi)    # MCTS.py:140
        cid, sampled_to = utils.decode_checker_index(sampled_index)
        sampled_from = root.state.checkers_pos[root.currPlayer][cid]
        sampled_edge = None
        for edge in root.edges:
            if edge.fromPos == sampled_from and edge.toPos == sampled_to:
                sampled_edge = edge
                break
        assert sampled_edge is not None
        return root.pi, sampled_edge
