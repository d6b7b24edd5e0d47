"""Gumbel search (gumbel=True / ccx_mcts_set_gumbel): self-play ply time against PUCT, and playing strength.

    python scripts/gumbel_bench.py --out DIR [--games 1024]

Writes DIR/r05_gumbel_bench.json with:
  selfplay   BatchedSelfPlay (accurate mode, 175 simulations, one leaf per round) at 180 and 4,096 slots, PUCT and Gumbel
             (m = 16) alternating twice, 7 warm-up plies then CUDA events around 3 plies; sims/s = slots x 175 / ply time
  strength   the same weights in two engines (accurate mode, train.evaluate's rules): Gumbel (m = 16, scale 1) at 175, 32 and
             16 simulations against PUCT at 175; colours swapped between two arenas of half the games each; win rate over
             decided games with a 95 % Wilson interval
The card's name and power limit are read by the same process."""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from leaves_bench import WEIGHTS, card, wilson  # noqa: E402
from reuse_bench import ply_ms  # noqa: E402
from chinesecheckersagent_b200.arena import BatchedArena  # noqa: E402
from chinesecheckersagent_b200.engine import Engine  # noqa: E402
from chinesecheckersagent_b200.model import ResidualCNN  # noqa: E402
from chinesecheckersagent_b200.selfplay import BatchedSelfPlay  # noqa: E402

SIMS = 175


def selfplay(model, eng):
    out = {}
    for n in (180, 4096):
        for rep in range(2):
            for gumbel in (False, True):
                sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=n, max_iters=32, gumbel=gumbel)
                for _ in range(7):
                    sp.step()
                ms = ply_ms(sp)
                key = "%d_%s" % (n, "gumbel" if gumbel else "puct")
                out.setdefault(key, []).append(dict(ms_per_ply=ms, sims_per_s=n * SIMS / ms * 1e3))
                print("self-play %d slots gumbel=%s: %.3f ms per ply" % (n, gumbel, ms), flush=True)
                del sp
    return out


def match(a, b, sims_a, games, seed):
    """Gumbel `a` at sims_a simulations against PUCT `b` at 175, `a` moving first in the first half of the games"""
    half = games // 2
    r1 = BatchedArena(a, b, half, seed=seed, enforce_move_limit=True, num_itr=(sims_a, SIMS), gumbel=(True, False)).play()
    r2 = BatchedArena(b, a, games - half, seed=seed, game_id0=half, enforce_move_limit=True, num_itr=(SIMS, sims_a),
                      gumbel=(False, True)).play()
    wins, losses = r1["p1_wins"] + r2["p2_wins"], r1["p2_wins"] + r2["p1_wins"]
    return dict(games=games, gumbel_simulations=sims_a, puct_simulations=SIMS, wins=wins, losses=losses,
                draws_or_unfinished=games - wins - losses, overflowed=r1["overflowed"] + r2["overflowed"],
                win_rate_of_decided=wins / (wins + losses) if wins + losses else None, wilson95=wilson(wins, wins + losses))


def strength(model, games, seed=2026):
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS).set_kernel("tc_acc")
    t0 = time.perf_counter()
    out = {}
    for k, sims in enumerate((175, 32, 16)):
        out["gumbel%d_vs_puct175" % sims] = r = match(model, other, sims, games, seed + k)
        print("Gumbel %d vs PUCT 175:" % sims, r, flush=True)
    out["seconds"] = time.perf_counter() - t0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--games", type=int, default=1024)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gumbel_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    eng = Engine(0)
    model = ResidualCNN(engine=eng).load_weights(WEIGHTS).set_kernel("tc_acc")
    res = dict(card=card(), simulations=SIMS, net_mode="tc_acc", gumbel=dict(considered=16, scale=1.0, c_visit=50.0, c_scale=0.1))
    res["selfplay"] = selfplay(model, eng)
    res["strength"] = strength(model, args.games)
    res["card_after"] = card()
    path = os.path.join(args.out, "r05_gumbel_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
