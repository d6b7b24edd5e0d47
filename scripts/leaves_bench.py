"""Leaf-parallel MCTS (leaves_per_round = L): drop-in decision latency, self-play rate and playing strength against L = 1.

    python scripts/leaves_bench.py --out DIR [--games 512]

Writes DIR/leaves_bench.json with:
  dropin     MCTS(Node(Board()), model, num_itr=175).search() in the accurate mode (tc_acc) for L in 1, 2, 4, 8, 16: 3 warm-up
             decisions, then a host clock around 20 decisions ending in a device synchronise (scripts/dropin_bench.py's method)
  selfplay   BatchedSelfPlay plies at 180, 1,024 and 4,096 slots for L in 1, 4, 8 (accurate mode): 7 warm-up plies, then CUDA
             events around 3 plies; sims/s = slots x 175 / ply time (scripts/selfplay_bench.py's figure)
  strength   the same weights in two engines, L = 8 against L = 1, colours alternating (half the games each way), and L = 8
             against the greedy player: train.evaluate's rules (tau = 0.01, move limit); win rate over decided games with a
             95 % Wilson interval
The card's name and power limit are read by the same process."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from chinesecheckersagent_b200.arena import GREEDY, BatchedArena  # noqa: E402
from chinesecheckersagent_b200.board import Board  # noqa: E402
from chinesecheckersagent_b200.engine import Engine  # noqa: E402
from chinesecheckersagent_b200.MCTS import MCTS, Node  # noqa: E402
from chinesecheckersagent_b200.model import ResidualCNN  # noqa: E402
from chinesecheckersagent_b200.selfplay import BatchedSelfPlay  # noqa: E402

WEIGHTS = os.path.join(ROOT, "tests", "golden", "good_model_weights.npz")
SIMS = 175


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    name, limit = [x.strip() for x in q.split(",")]
    return dict(name=name, power_limit=limit)


def wilson(k, n, z=1.96):
    if n == 0:
        return None
    p = k / n
    d = 1 + z * z / n
    c = (p + z * z / (2 * n)) / d
    h = z * math.sqrt(p * (1 - p) / n + z * z / (4 * n * n)) / d
    return [c - h, c + h]


def dropin(model, eng, reps=20):
    out = {}
    model.set_kernel("tc_acc")
    old = MCTS.LEAVES_PER_ROUND
    try:
        for L in (1, 2, 4, 8, 16):
            MCTS.LEAVES_PER_ROUND = L
            f = lambda: MCTS(Node(Board(engine=eng), 1), model, num_itr=SIMS).search()   # noqa: E731
            for _ in range(3):
                f()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                f()
            torch.cuda.synchronize()
            out[str(L)] = dict(ms_per_decision=(time.perf_counter() - t0) / reps * 1e3, rounds=1 + (SIMS - 1 + L - 1) // L)
            print("drop-in L=%d: %.3f ms" % (L, out[str(L)]["ms_per_decision"]), flush=True)
    finally:
        MCTS.LEAVES_PER_ROUND = old
    return out


def selfplay(model, eng, reps=3):
    out = {}
    model.set_kernel("tc_acc")
    for n in (180, 1024, 4096):
        for L in (1, 4, 8):
            sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=n, max_iters=32, leaves_per_round=L)
            for _ in range(7):
                sp.step()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                sp.step()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps
            out["%d_L%d" % (n, L)] = dict(slots=n, leaves=L, ms_per_ply=ms, sims_per_s=n * SIMS / ms * 1e3)
            print("self-play %d slots L=%d: %.3f ms per ply, %.4g sims/s" % (n, L, ms, n * SIMS / ms * 1e3), flush=True)
            del sp
    return out


def match(a, b, la, lb, games, seed):
    """a (leaves la) against b (leaves lb), a moving first in the first half of the games, second in the other half"""
    half = games // 2
    r1 = BatchedArena(a, b, half, seed=seed, enforce_move_limit=True, leaves_per_round=(la, lb)).play()
    r2 = BatchedArena(b, a, games - half, seed=seed, game_id0=half, enforce_move_limit=True, leaves_per_round=(lb, la)).play()
    wins, losses = r1["p1_wins"] + r2["p2_wins"], r1["p2_wins"] + r2["p1_wins"]
    return dict(games=games, wins=wins, losses=losses, draws_or_unfinished=games - wins - losses,
                win_rate_of_decided=wins / (wins + losses) if wins + losses else None, wilson95=wilson(wins, wins + losses))


def strength(model, games, seed=2026):
    model.set_kernel("tc_acc")
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS).set_kernel("tc_acc")
    t0 = time.perf_counter()
    vs_one = match(model, other, 8, 1, games, seed)
    print("L=8 vs L=1:", vs_one, flush=True)
    vs_greedy = match(model, GREEDY, 8, 1, games, seed + 1)
    print("L=8 vs greedy:", vs_greedy, flush=True)
    return dict(l8_vs_l1=vs_one, l8_vs_greedy=vs_greedy, seconds=time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--games", type=int, default=512)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("leaves_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    eng = Engine(0)
    model = ResidualCNN(engine=eng).load_weights(WEIGHTS)
    res = dict(card=card(), simulations=SIMS, net_mode="tc_acc")
    res["dropin"] = dropin(model, eng)
    res["selfplay"] = selfplay(model, eng)
    res["strength"] = strength(model, args.games)
    res["card_after"] = card()
    path = os.path.join(args.out, "leaves_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
