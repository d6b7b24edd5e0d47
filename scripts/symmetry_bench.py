"""Mirror-symmetric net evaluation (ResidualCNN.set_symmetry / ccx_net_set_symmetry): self-play ply time and playing strength.

    python scripts/symmetry_bench.py --out DIR [--games 1024]

Writes DIR/r05_symmetry_bench.json with:
  selfplay   BatchedSelfPlay (accurate mode, 175 simulations, one leaf per round) at 180 and 4,096 slots with the symmetry off,
             random and mean, alternating twice, 7 warm-up plies then CUDA events around 3 plies; sims/s = slots x 175 / ply time
  strength   the same weights in two engines (accurate mode, train.evaluate's rules, random PUCT ties): random at 175 simulations
             and mean at 175, 88 and 44 against off at 175; colours swapped between two arenas of half the games each; win rate
             over decided games with a 95 % Wilson interval
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
SEED = 0x5EED


def selfplay(model, eng):
    out = {}
    for n in (180, 4096):
        for rep in range(2):
            for mode in ("off", "random", "mean"):
                model.set_symmetry(mode, SEED)
                sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=n, max_iters=32)
                for _ in range(7):
                    sp.step()
                ms = ply_ms(sp)
                out.setdefault("%d_%s" % (n, mode), []).append(dict(ms_per_ply=ms, sims_per_s=n * SIMS / ms * 1e3))
                print("self-play %d slots symmetry=%s: %.3f ms per ply" % (n, mode, ms), flush=True)
                del sp
    model.set_symmetry("off")
    return out


def match(a, b, mode, sims_a, games, seed):
    """`a` with the symmetry `mode` at sims_a simulations against `b` with it off at 175, `a` moving first in the first half"""
    a.set_symmetry(mode, SEED)
    b.set_symmetry("off")
    half = games // 2
    r1 = BatchedArena(a, b, half, seed=seed, enforce_move_limit=True, num_itr=(sims_a, SIMS)).play()
    r2 = BatchedArena(b, a, games - half, seed=seed, game_id0=half, enforce_move_limit=True, num_itr=(SIMS, sims_a)).play()
    a.set_symmetry("off")
    wins, losses = r1["p1_wins"] + r2["p2_wins"], r1["p2_wins"] + r2["p1_wins"]
    return dict(games=games, symmetry=mode, simulations=sims_a, off_simulations=SIMS, wins=wins, losses=losses,
                draws_or_unfinished=games - wins - losses, overflowed=r1["overflowed"] + r2["overflowed"],
                win_rate_of_decided=wins / (wins + losses) if wins + losses else None, wilson95=wilson(wins, wins + losses))


def strength(model, games, seed=2026):
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS).set_kernel("tc_acc")
    t0 = time.perf_counter()
    out = {}
    for k, (mode, sims) in enumerate((("random", 175), ("mean", 175), ("mean", 88), ("mean", 44))):
        out["%s%d_vs_off175" % (mode, sims)] = r = match(model, other, mode, sims, games, seed + k)
        print("%s %d vs off 175:" % (mode, sims), r, flush=True)
    out["seconds"] = time.perf_counter() - t0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--games", type=int, default=1024)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("symmetry_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    eng = Engine(0)
    model = ResidualCNN(engine=eng).load_weights(WEIGHTS).set_kernel("tc_acc")
    res = dict(card=card(), simulations=SIMS, net_mode="tc_acc", orientation_seed=SEED)
    res["selfplay"] = selfplay(model, eng)
    res["strength"] = strength(model, args.games)
    res["card_after"] = card()
    path = os.path.join(args.out, "r05_symmetry_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
