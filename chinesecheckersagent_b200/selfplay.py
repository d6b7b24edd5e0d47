"""Batched selfplay.selfplay() (selfplay.py:11-133): n game slots per GPU advance one ply per iteration;
opening plies are random (INITIAL_RANDOM_MOVES), later plies run a full MCTS (root pre-expanded, Dirichlet
noise, MCTS_SIMULATIONS simulations) for every slot at once with ONE batched net evaluation per simulation
round.  Finished games are labelled / discarded on the device and their slot restarts immediately.

`collect()` returns the trajectory in utils.convert_to_train_data's format: board_x (N,7,7,7), pi_y (N,294),
v_y (N,); `all_gather()` merges the per-rank buffers over NCCL (the only collective in the system)."""
import torch

from .config import (C_PUCT, DEFAULT_SEED, DIRICHLET_ALPHA, DTYPE_U8, INITIAL_RANDOM_MOVES, MCTS_SIMULATIONS,
                     PROGRESS_MOVE_LIMIT, STATE_WORDS, TOTAL_MOVES_TILL_TAU0)
from .engine import MAX_LEAVES, REUSE_CARRY, BatchedEnv, _p

NOISE_STRIDE = 128


class UniformEvaluator:
    """Stub evaluator of BASELINE configs[3]: p = 1/294 everywhere, v = 0.0."""

    def __init__(self, engine, n):
        self.p = torch.full((n, 294), 1 / 294., dtype=torch.float64, device=engine.device)
        self.v = torch.zeros((n,), dtype=torch.float64, device=engine.device)

    def __call__(self, leaf_state):
        return self.p, self.v


class BatchedSelfPlay:
    """n game slots advancing one ply per `step()`.

    evaluate      ResidualCNN.evaluate_states of a model living in `engine` (fused C round loop, ccx_mcts_run_net) or any
                  callable leaf_state (5, n) -> (p (n, 294) float64, v (n,) float64) (one round trip per simulation)
    opponent      a second loaded ResidualCNN in its OWN Engine on the same GPU: two-net self-play (selfplay.py:11-29,58 —
                  model1 decides on even plies, model2 on odd ones; train.py:62 other_opponent_for_selfplay)
    random_ties   PUCT ties drawn uniformly among the reference's epsilon-tie list (MCTS.py:65-72) with Philox; False = first
                  maximal edge, the bit-exact parity mode the oracle tests use
    ring          record buffers are a ring over iterations: games longer than max_iters // 2 iterations are discarded
                  (status OVERFLOW) and finished records are moved out every max_iters // 2 iterations, so the loop can run
                  for as long as the caller wants; False = the buffers hold exactly max_iters iterations and step() raises after
    leaves_per_round  L > 1: each search round selects up to L leaves per tree under virtual loss and evaluates n*L positions
                  at once (include/ccx.h, ccx_mcts_run_net_leaves; `evaluate` then receives (5, n*L) leaf states): about
                  1 + num_itr / L rounds per ply instead of num_itr + 1.  1 (default) = one simulation per tree per round
    reuse_tree    each ply's search starts from the subtree the slot's previous search grew below the move that was played
                  (include/ccx.h, ccx_mcts_begin_reuse; at most reuse_carry times one search's nodes, edges and visits), the
                  Dirichlet noise mixed into the carried root's priors; stats() then counts reused and fresh searches.  Not with
                  `opponent` (each net's trees would skip every other ply)
    gumbel        Gumbel search (BatchedMCTS gumbel=True; gumbel_considered, gumbel_scale, gumbel_c_visit, gumbel_c_scale as there,
                  the draws keyed by the slot ids): no Dirichlet noise (the Gumbel draws are the exploration), the move played is
                  the search's action, the record's policy target is the improved policy.  Not with `opponent`, leaves_per_round > 1
                  or reuse_tree
    """

    def __init__(self, engine, evaluate, n_slots=4096, seed=DEFAULT_SEED, rank=0, world=1, num_itr=MCTS_SIMULATIONS,
                 cpuct=C_PUCT, max_iters=256, edges_per_tree=0, dirichlet=True, log_moves=False, fused=None, ring=False,
                 random_ties=True, opponent=None, leaves_per_round=1, reuse_tree=False, reuse_carry=REUSE_CARRY, gumbel=False,
                 gumbel_considered=16, gumbel_scale=1.0, gumbel_c_visit=50.0, gumbel_c_scale=0.1):
        self.eng, self.evaluate = engine, evaluate
        owner = getattr(evaluate, "__self__", None)
        auto = getattr(owner, "fused_mcts", False) and getattr(owner, "eng", None) is engine and getattr(evaluate, "__name__", "") == "evaluate_states"
        self.fused = bool(auto) if fused is None else bool(fused)
        self.n, self.seed, self.rank, self.world = int(n_slots), int(seed), int(rank), int(world)
        self.n0 = self.n                                 # slots at construction: RNG keys use rank * n0 + original slot index, compaction or not
        self.num_itr, self.cpuct, self.max_iters, self.ept = int(num_itr), float(cpuct), int(max_iters), int(edges_per_tree)
        self.dirichlet, self.ring, self.random_ties = dirichlet, bool(ring), bool(random_ties)
        self.opponent = opponent
        self.leaves = int(leaves_per_round)
        if not 1 <= self.leaves <= MAX_LEAVES:
            raise ValueError("leaves_per_round must be in 1..%d" % MAX_LEAVES)
        self.reuse_tree, self.reuse_carry = bool(reuse_tree), int(reuse_carry)
        if self.reuse_tree and opponent is not None:
            raise ValueError("reuse_tree is not supported with two-net self-play (opponent=)")
        if self.reuse_carry < 0:
            raise ValueError("reuse_carry must be >= 0")
        self.gumbel = bool(gumbel)
        if self.gumbel:
            if opponent is not None or self.leaves != 1 or self.reuse_tree:
                raise ValueError("Gumbel self-play has one net, one leaf per round and fresh trees (no opponent, leaves_per_round, reuse_tree)")
            self.dirichlet = False
            self.gumbel_params = (int(gumbel_considered), float(gumbel_scale), float(gumbel_c_visit), float(gumbel_c_scale),
                                  (self.seed ^ 0x6B3E1) & 0xFFFFFFFFFFFFFFFF)
            if self.gumbel_params[0] < 1 or min(self.gumbel_params[1:4]) < 0:
                raise ValueError("gumbel_considered must be >= 1 and the Gumbel scales >= 0")
        if opponent is not None:
            if not self.fused:
                raise ValueError("two-net self-play needs `evaluate` to be the evaluate_states of a ResidualCNN in `engine`")
            if opponent.eng is engine:
                raise ValueError("the opponent net needs its own Engine (one set of net weights per ccx handle)")
        e, n = engine, self.n
        self.env = BatchedEnv(n, engine=e, seed=seed, game_id0=rank * n)
        self.leaf = e.empty((5, n * self.leaves), torch.int64)
        self.noise = e.empty((n, NOISE_STRIDE), torch.float64)
        self.visits = e.empty((n, 294), torch.int32)
        self.tree_nodes = e.empty((n,), torch.int32)
        if opponent is not None:
            self.visits2 = e.empty((n, 294), torch.int32)
            self.tree_nodes2 = e.empty((n,), torch.int32)
        self.serial = e.zeros((n,), torch.int64)
        self.start_iter = e.zeros((n,), torch.int32)
        self.counters = e.zeros((8,), torch.int64)
        self.reused = e.empty((n,), torch.int32) if self.reuse_tree else None
        self.reuse_counts = e.zeros((2,), torch.int64) if self.reuse_tree else None     # searches carried / started fresh
        self._prev = None                                # after compact(): previous slot of every kept slot, for the next search
        self.starts_left = None                          # device int64[1] once play_games() set a budget of game starts
        self.rec_state = e.zeros((self.max_iters * n, 5), torch.int64)
        self.rec_visits = e.zeros((self.max_iters * n, 294), torch.int16)
        self.rec_flag = e.zeros((self.max_iters * n,), torch.uint8)
        if self.gumbel:
            self.pi = e.empty((n, 294), torch.float64)
            self.action = e.empty((n,), torch.int32)
            self.rec_pi = e.zeros((self.max_iters * n, 294), torch.float32)
        self.move_log = e.zeros((self.max_iters * n,), torch.int32) if log_moves else None
        self.slot_ids = torch.arange(rank * n, (rank + 1) * n, dtype=torch.int64, device=e.device)     # global identity of every slot
        self.compactions = 0
        self.iter = 0
        self._last_collect = 0
        self._chunks = []

    @property
    def max_game_iters(self):
        return max(2, self.max_iters // 2) if self.ring else self.max_iters

    def _search(self, eng, parity, visits, tree_nodes):
        """one full search of every slot whose mover uses the net living in `eng` (parity -1: all slots)"""
        n, st = self.n, self.env.state
        eng.call("ccx_set_slot_ids", _p(self.slot_ids))
        eng.call("ccx_mcts_set_tiebreak", 1 if self.random_ties else 0, self.seed ^ 0x71E5, self.rank * self.n0)
        if self.gumbel:
            self._search_gumbel(eng, visits, tree_nodes)
            return
        if self.reuse_tree:
            eng.call("ccx_mcts_begin_reuse", n, _p(st), self.num_itr + 1, self.ept, INITIAL_RANDOM_MOVES, parity, self.reuse_carry,
                     _p(self._prev), _p(self.noise) if self.dirichlet else None, NOISE_STRIDE, 1, _p(self.reused))
            self._prev = None
            self.reuse_counts += torch.stack([(self.reused > 0).sum(), (self.reused == 0).sum()])
        else:
            eng.call("ccx_mcts_begin", n, _p(st), self.num_itr + 1, self.ept, INITIAL_RANDOM_MOVES, parity)
        L = self.leaves
        if self.fused and L > 1:
            eng.call("ccx_mcts_run_net_leaves", n, self.num_itr + 1, L, self.cpuct, _p(self.noise) if self.dirichlet else None,
                     NOISE_STRIDE, 1)
        elif self.fused:                                 # the library's own net: all rounds in one C call, fused round kernels
            eng.call("ccx_mcts_run_net", n, self.num_itr + 1, self.cpuct, _p(self.noise) if self.dirichlet else None,
                     NOISE_STRIDE, 1)
        elif L > 1:                                      # round 0 = the root expansion, then up to L leaves per round
            eng.call("ccx_mcts_leaf_budget", n, L, self.num_itr + 1)
            for r in range(1 + (self.num_itr + L - 1) // L):
                eng.call("ccx_mcts_select_leaves", n, L, self.cpuct, _p(self.leaf))
                p, v = self.evaluate(self.leaf)
                noise = self.noise if (r == 0 and self.dirichlet) else None
                eng.call("ccx_mcts_expand_backup_leaves", n, L, _p(p), _p(v), _p(noise), NOISE_STRIDE if noise is not None else 0, 1)
        else:
            for r in range(self.num_itr + 1):           # round 0 = make_move's root expansion (selfplay.py:117)
                eng.call("ccx_mcts_select", n, self.cpuct, _p(self.leaf))
                p, v = self.evaluate(self.leaf)
                noise = self.noise if (r == 0 and self.dirichlet) else None
                eng.call("ccx_mcts_expand_backup", n, _p(p), _p(v), _p(noise), NOISE_STRIDE if noise is not None else 0, 1)
        eng.call("ccx_mcts_finalize", n, 1.0, _p(visits), None, None, _p(tree_nodes))
        eng.call("ccx_set_slot_ids", None)               # other users of this engine identify their trees by position again

    def _search_gumbel(self, eng, visits, tree_nodes):
        """the Gumbel search of every slot; visits becomes the one-hot row of the chosen action (the sampler of
        ccx_selfplay_advance then plays exactly that move: the row's only non-zero weight, 1 or 1^(1/tau) = 1, covers the
        whole interval [0, 1) a uniform draw falls into, for every draw and every tau)"""
        n, st = self.n, self.env.state
        eng.call("ccx_mcts_set_gumbel", 1, *self.gumbel_params)
        try:
            eng.call("ccx_mcts_begin", n, _p(st), self.num_itr + 1, self.ept, INITIAL_RANDOM_MOVES, -1)
            if self.fused:
                eng.call("ccx_mcts_run_net", n, self.num_itr + 1, self.cpuct, None, 0, 0)
            else:
                for _ in range(self.num_itr + 1):       # round 0 = the root expansion
                    eng.call("ccx_mcts_select", n, self.cpuct, _p(self.leaf))
                    p, v = self.evaluate(self.leaf)
                    eng.call("ccx_mcts_expand_backup", n, _p(p), _p(v), None, 0, 0)
            eng.call("ccx_mcts_finalize_gumbel", n, _p(visits), _p(self.pi), None, _p(self.action), _p(tree_nodes))
        finally:
            eng.call("ccx_mcts_set_gumbel", 0, 1, 0.0, 0.0, 0.0, 0)
            eng.call("ccx_set_slot_ids", None)
        visits.zero_()
        act = self.action.long()
        visits.scatter_(1, act.clamp(min=0).unsqueeze(1), (act >= 0).int().unsqueeze(1))

    # one ply for every slot
    def step(self, restart=True):
        e, n, it = self.eng, self.n, self.iter
        if not self.ring and it >= self.max_iters:
            raise RuntimeError("record buffer full after max_iters = %d iterations: construct with ring=True (or a larger max_iters)"
                               % self.max_iters)
        uid0 = self.rank * self.n0
        st = self.env.state
        e.call("ccx_set_slot_ids", _p(self.slot_ids))
        if self.dirichlet:
            e.call("ccx_gamma_noise", n, NOISE_STRIDE, DIRICHLET_ALPHA, self.seed, it, uid0, _p(self.noise))
        if self.opponent is None:
            self._search(e, -1, self.visits, self.tree_nodes)
            visits, tree_nodes = self.visits, self.tree_nodes
        else:
            # selfplay.py:29,58: model1 on even plies, model2 on odd ones; each net searches its own slots (the other slots get
            # an inactive tree: zero visits, node count -2), both on torch's current stream
            self._search(e, 0, self.visits, self.tree_nodes)
            self._search(self.opponent.eng, 1, self.visits2, self.tree_nodes2)
            visits = self.visits + self.visits2
            tree_nodes = torch.where(self.tree_nodes == -2, self.tree_nodes2, self.tree_nodes)
        e.call("ccx_set_slot_ids", _p(self.slot_ids))
        e.call("ccx_selfplay_advance", n, _p(st), _p(visits), _p(tree_nodes), self.seed, it, uid0, _p(self.serial),
               self.world * self.n0, INITIAL_RANDOM_MOVES, TOTAL_MOVES_TILL_TAU0, PROGRESS_MOVE_LIMIT, _p(self.rec_state),
               _p(self.rec_visits), _p(self.rec_flag), self.max_iters, _p(self.counters), _p(self.move_log))
        if self.gumbel:
            e.call("ccx_selfplay_record_pi", n, it, _p(self.pi), _p(self.rec_pi), self.max_iters)
        e.call("ccx_selfplay_finish", n, _p(st), it, _p(self.start_iter), _p(self.serial), _p(self.rec_state),
               _p(self.rec_flag), self.max_iters, self.max_game_iters if self.ring else 0, int(bool(restart)),
               _p(self.starts_left), _p(self.counters))
        e.call("ccx_set_slot_ids", None)
        self.iter += 1
        if self.ring and self.iter - self._last_collect >= self.max_iters - self.max_game_iters:
            self._drain()

    def running(self):
        return int(((self.env.state[4] >> 56) == 0).sum().item())

    def compact(self):
        """Drop the slots whose game has ended and may not restart (the drain of play_games): the batch every kernel and the
        net sees shrinks to the games still running, which continue bit for bit as they would have (their Philox streams are
        keyed by `slot_ids`, not by position).  Finished records are moved out first.  Returns the new slot count."""
        self._drain()
        keep = torch.nonzero((self.env.state[4] >> 56) == 0).flatten()
        m, n, R, e = int(keep.numel()), self.n, self.max_iters, self.eng
        if m == 0 or m == n:
            return n
        by_iter = lambda t: t.view(R, n, *t.shape[1:])[:, keep].reshape(R * m, *t.shape[1:]).contiguous()
        self.rec_state, self.rec_visits, self.rec_flag = by_iter(self.rec_state), by_iter(self.rec_visits), by_iter(self.rec_flag)
        if self.gumbel:
            self.rec_pi = by_iter(self.rec_pi)
            self.pi, self.action = e.empty((m, 294), torch.float64), e.empty((m,), torch.int32)
        if self.move_log is not None:
            self.move_log = by_iter(self.move_log)
        state = self.env.state[:, keep].contiguous()
        self.env = BatchedEnv(m, engine=e, seed=self.seed, game_id0=self.rank * self.n0, state=state)
        self.serial, self.start_iter, self.slot_ids = (self.serial[keep].contiguous(), self.start_iter[keep].contiguous(),
                                                       self.slot_ids[keep].contiguous())
        self.n = m
        self.leaf = e.empty((5, m * self.leaves), torch.int64)
        self.noise = e.empty((m, NOISE_STRIDE), torch.float64)
        self.visits, self.tree_nodes = e.empty((m, 294), torch.int32), e.empty((m,), torch.int32)
        if self.reuse_tree:
            self.reused = e.empty((m,), torch.int32)
            self._prev = keep if self._prev is None else self._prev[keep]
        if self.opponent is not None:
            self.visits2, self.tree_nodes2 = e.empty((m, 294), torch.int32), e.empty((m,), torch.int32)
        self.compactions += 1
        return m

    def stats(self):
        c = self.counters.cpu().tolist()
        out = dict(plies=c[0], p1_wins=c[1], p2_wins=c[2], discarded_repetition=c[3], discarded_no_progress=c[4],
                   discarded_overflow=c[5], records=c[6], games=c[7], iterations=self.iter)
        if self.reuse_tree:
            out["reused_searches"], out["fresh_searches"] = self.reuse_counts.cpu().tolist()
        return out

    def run(self, target_games=None, iters=None, poll_every=8):
        """Throughput loop: every finished slot restarts at once, stop after `iters` iterations or once `target_games` games
        were kept.  Stopping on a count of FINISHED games favours short games (long ones are still in flight when the loop
        ends); `play_games()` is the reference's semantics (exactly N games started, all played out)."""
        done = 0
        while True:
            self.step()
            done += 1
            if iters is not None and done >= iters:
                break
            if not self.ring and self.iter >= self.max_iters:
                break
            if target_games is not None and done % poll_every == 0 and self.stats()["games"] >= target_games:
                break
        out = self.stats()
        if target_games is not None and out["games"] < target_games:
            import warnings
            warnings.warn("BatchedSelfPlay.run stopped after %d iterations with %d of the %d requested games"
                          % (done, out["games"], target_games), RuntimeWarning)
        return out

    def play_games(self, num_games, poll_every=8, max_iterations=None, compact=True, compact_min=256, compact_ratio=0.75):
        """train.generate_self_play's contract (train.py:58-64): exactly `num_games` games are STARTED, every one of them is
        played to its end (win, or discarded by the repetition / progress rules), nothing else is recorded.  Slots restart
        while the budget of starts lasts, then drain; during the drain the batch is compacted whenever no more than `compact_ratio` of its
        slots are still playing (`compact_ratio`; `compact=False` keeps the full batch: same games, same records).  Returns stats(); the records
        are in collect()."""
        if self.iter != 0:
            raise RuntimeError("play_games() needs a fresh BatchedSelfPlay")
        self.ring = True
        n, num_games = self.n, int(num_games)
        active = min(n, num_games)
        if active < n:                                   # fewer games than slots: the surplus slots never play
            from .config import ST_NO_MOVES
            self.env.state[4, active:] |= (ST_NO_MOVES << 56)
            self.start_iter[active:] = 0x7FFFFFFF
        self.starts_left = torch.tensor([num_games - active], dtype=torch.int64, device=self.eng.device)
        cap = max_iterations or (2 + (num_games + n - 1) // n) * self.max_game_iters
        while self.iter < cap:
            self.step()
            if self.iter % poll_every == 0:
                live = self.running()
                if live == 0:
                    break
                if compact and live <= compact_ratio * self.n and self.n > compact_min and int(self.starts_left.item()) <= 0:
                    self.compact()
        out = self.stats()
        out["unfinished"] = self.running()
        out["compactions"] = self.compactions
        out["games_started"] = num_games - max(0, int(self.starts_left.item()))
        return out

    # trajectory in utils.convert_to_train_data's format (utils.py:60-73)
    def _pack_finished(self):
        """labelled records -> dict of device tensors; the records are consumed (their flags return to 0)"""
        e = self.eng
        flags = self.rec_flag & 0xF
        rows = torch.nonzero((flags == 2) | (flags == 3)).flatten().contiguous()
        m = int(rows.numel())
        out_state = e.empty((5, max(m, 1)), torch.int64)
        pi_y = e.empty((m, 294), torch.float32)
        v_y = e.empty((m,), torch.int8)
        board_x = e.empty((m, 7, 7, 7), torch.uint8)
        if m:
            e.call("ccx_traj_pack_pi" if self.gumbel else "ccx_traj_pack", m, _p(rows), _p(self.rec_state),
                   _p(self.rec_pi if self.gumbel else self.rec_visits), _p(self.rec_flag), _p(out_state), _p(pi_y), _p(v_y))
            e.call("ccx_encode", m, _p(out_state), _p(board_x), DTYPE_U8)
            self.rec_flag[rows] = 0
        return dict(board_x=board_x, pi_y=pi_y, v_y=v_y, state=out_state[:, :m].contiguous())

    def _drain(self):
        chunk = self._pack_finished()
        if chunk["v_y"].shape[0]:
            self._chunks.append(chunk)
        self._last_collect = self.iter

    def collect(self):
        """Every record of a finished, kept game since the last collect(): board_x (M,7,7,7) uint8, pi_y (M,294) float32,
        v_y (M,) int8, state (5,M) packed words.  Consuming: a second call returns only what finished in between."""
        self._drain()
        chunks, self._chunks = self._chunks, []
        if not chunks:
            return self._pack_finished()
        if len(chunks) == 1:
            return chunks[0]
        return dict(board_x=torch.cat([c["board_x"] for c in chunks]), pi_y=torch.cat([c["pi_y"] for c in chunks]),
                    v_y=torch.cat([c["v_y"] for c in chunks]), state=torch.cat([c["state"] for c in chunks], dim=1))


def all_gather_trajectories(traj, group=None):
    """NCCL (or gloo) all-gather of the per-rank trajectory buffers into the training buffer (train.py:88-92 collects the
    workers' pickled game lists the same way); ranks hold different numbers of records, so counts are gathered first and
    the buffers padded to the maximum.  Keys: board_x, pi_y, v_y and, when present, the packed `state` words."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return traj
    world = dist.get_world_size(group)
    dev = traj["board_x"].device
    m = torch.tensor([traj["board_x"].shape[0]], dtype=torch.int64, device=dev)
    counts = torch.zeros(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(counts, m, group=group)
    counts = counts.cpu().tolist()                      # the one host sync: the output sizes depend on it
    mx = max(max(counts), 1)
    out = {"counts": counts}
    src = dict(traj)
    if "state" in src:
        src["state"] = src["state"].t().contiguous()    # (5, M) plane-major -> (M, 5) records
    for key in ("board_x", "pi_y", "v_y", "state"):
        if key not in src:
            continue
        t = src[key]
        pad = torch.zeros((mx,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        pad[:t.shape[0]] = t
        full = torch.empty((world * mx,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
        dist.all_gather_into_tensor(full, pad, group=group)
        out[key] = torch.cat([full[r * mx:r * mx + counts[r]] for r in range(world)], dim=0)
    if "state" in out:
        out["state"] = out["state"].t().contiguous()
    return out


def check_gathered_trajectories(engine, local, gathered, group=None, sample=4096):
    """Consistency of an all-gathered training buffer, asserted on every rank: the gathered count is the sum of the ranks'
    counts, this rank's slice is its own local buffer, every rank holds the same bytes (a checksum of board_x / pi_y / v_y is
    compared across ranks), v_y is +-1 and pi_y is supported on legal moves of the recorded position (movegen on a sample).
    Returns the figures it checked."""
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    counts = gathered.get("counts", [int(local["v_y"].shape[0])])
    total = int(gathered["v_y"].shape[0])
    assert total == sum(counts) and counts[rank] == int(local["v_y"].shape[0]), (counts, total)
    lo = sum(counts[:rank])
    for key in ("board_x", "pi_y", "v_y"):
        assert torch.equal(gathered[key][lo:lo + counts[rank]], local[key]), "rank %d: its own slice of %s changed in the gather" % (rank, key)
    v = gathered["v_y"]
    assert bool(((v == 1) | (v == -1)).all())
    pi = gathered["pi_y"]
    assert bool((pi >= 0).all()) and bool(((pi.double().sum(1) - 1).abs() < 1e-4).all())
    checksum = torch.stack([gathered["board_x"].sum(dtype=torch.int64).double(), (pi.double() * torch.arange(1, 295, device=pi.device)).sum(),
                            v.sum(dtype=torch.int64).double(), torch.tensor(float(total), device=pi.device, dtype=torch.float64)])
    if world > 1:
        sums = torch.empty((world, 4), dtype=torch.float64, device=pi.device)
        dist.all_gather_into_tensor(sums, checksum.unsqueeze(0).contiguous(), group=group)
        assert bool((sums == sums[0:1]).all()), "ranks hold different gathered buffers: %s" % sums.tolist()
    checked = 0
    if "state" in gathered and total:
        idx = torch.linspace(0, total - 1, min(sample, total), device=pi.device).long()
        st = torch.zeros((STATE_WORDS, idx.numel()), dtype=torch.int64, device=pi.device)
        st[:5] = gathered["state"][:, idx]
        masks = BatchedEnv(idx.numel(), engine=engine, state=st).movegen()                      # (6, k) destination bitboards
        a = torch.arange(294, device=pi.device)
        cid, off = a // 49, a % 49
        bit = (off // 7) * 8 + off % 7
        legal = ((masks[cid, :].t() >> bit) & 1).bool()                                          # (k, 294)
        assert not bool(((pi[idx] > 0) & ~legal).any()), "pi_y has mass on an illegal move"
        checked = int(idx.numel())
    return dict(records_total=total, counts=counts, checksum=checksum.tolist(), legal_support_checked=checked)


# ---- selfplay.selfplay(model1, model2=None, randomised=False), one game, same contract as selfplay.py:11-80 ----
def selfplay(model1, model2=None, randomised=False, num_itr=MCTS_SIMULATIONS):
    """Returns (play_history [(Board, pi)], reward for player 1) or (None, None) for a discarded game; what
    train.py:62 calls.  For throughput use BatchedSelfPlay; this mirror exists for drop-in compatibility."""
    import copy
    import random

    import numpy as np

    from . import utils
    from .board import Board
    from .config import (BOARD_HIST_MOVES, DET_TREE_TAU, DIR_NOISE_FACTOR, NUM_CHECKERS, PLAYER_ONE, PLAYER_TWO,
                         TOTAL_HIST_MOVES, TREE_TAU, UNIQUE_DEST_LIMIT)
    from .MCTS import MCTS, Node
    model2 = model2 or model1
    player_progresses, player_turn, num_useless_moves, play_history, tree_tau = [0, 0], 0, 0, [], TREE_TAU
    root = Node(Board(randomised=randomised, engine=getattr(model1, "eng", None)), PLAYER_ONE)     # the model's device, not cuda:0
    use_model1 = True
    while True:
        model = model1 if use_model1 else model2
        if len(root.state.hist_moves) < INITIAL_RANDOM_MOVES:                       # selfplay.py:32-33, 83-104
            valid = root.state.get_valid_moves(root.currPlayer)
            start = random.choice([k for k in valid if valid[k]])
            nxt = copy.deepcopy(root.state)
            nxt.place(root.currPlayer, start, random.choice(valid[start]))
            root = Node(nxt, PLAYER_ONE + PLAYER_TWO - root.currPlayer)
        else:                                                                       # selfplay.py:107-133
            tree = MCTS(root, model, num_itr=num_itr, tree_tau=tree_tau)
            tree.expandAndBackUp(tree.root, breadcrumbs=[])
            noise = np.random.dirichlet(np.ones(len(tree.root.edges)) * DIRICHLET_ALPHA)
            for i, e in enumerate(tree.root.edges):
                e.stats['P'] *= (1. - DIR_NOISE_FACTOR)
                e.stats['P'] += DIR_NOISE_FACTOR * noise[i]
            pi, edge = tree.search()
            play_history.append((tree.root.state, pi))
            root = Node(copy.deepcopy(edge.outNode.state), edge.outNode.currPlayer)
        hm = root.state.hist_moves
        mine = [hm[i] for i in range(len(hm) - 1, -1, -2)]
        if len(mine) * 2 >= TOTAL_HIST_MOVES and len(set(m[1] for m in mine)) <= UNIQUE_DEST_LIMIT:
            return None, None                                                       # selfplay.py:45-47
        progress = root.state.player_progress(player_turn + 1)
        if progress > player_progresses[player_turn]:
            num_useless_moves = int(num_useless_moves * (NUM_CHECKERS - 1) / NUM_CHECKERS)
            player_progresses[player_turn] = progress
        else:
            num_useless_moves += 1
        player_turn, use_model1 = 1 - player_turn, not use_model1
        if len(play_history) + INITIAL_RANDOM_MOVES > TOTAL_MOVES_TILL_TAU0:
            tree_tau = DET_TREE_TAU
        if root.state.check_win():
            break
        if num_useless_moves >= PROGRESS_MOVE_LIMIT:
            return None, None
    reward = utils.get_p1_winloss_reward(root.state)
    return (play_history[BOARD_HIST_MOVES:] if randomised else play_history), reward
