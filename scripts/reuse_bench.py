"""Tree reuse (reuse_tree / ccx_mcts_begin_reuse): cost of the reuse begin, self-play rate with and without it, how much it
carries, pool bytes, and playing strength.

    python scripts/reuse_bench.py --out DIR [--games 1024]

Writes DIR/reuse_bench.json with:
  begin      self-play (accurate mode, one leaf per round, reuse on) at 4,096 and 7,104 slots after 8 warm-up plies: per-ply
             device time of k_mcts_reuse_match / _gather / _commit from torch.profiler over 3 plies, against the ply time
             (CUDA events around 3 plies of a run without the profiler)
  selfplay   BatchedSelfPlay plies at 180 and 4,096 slots with reuse off and on, alternating, 7 warm-up plies then CUDA events
             around 3 plies; sims/s = slots x 175 / ply time
  carried    1,024 slots started together, reuse on: per iteration the share of active searches that carried a tree and the
             mean root visits the carried trees brought along (root visits after the search - 176)
  pool       ccx_mcts_pool_bytes at 4,096 slots with reuse off and on
  strength   the same weights in two engines (accurate mode, 175 simulations, train.evaluate's rules): reuse against no reuse
             at L = 1, and L = 8 with reuse against L = 1 without; colours swapped between two arenas of half the games each;
             win rate over decided games with a 95 % Wilson interval
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
from chinesecheckersagent_b200.arena import BatchedArena  # noqa: E402
from chinesecheckersagent_b200.engine import Engine  # noqa: E402
from chinesecheckersagent_b200.model import ResidualCNN  # noqa: E402
from chinesecheckersagent_b200.selfplay import BatchedSelfPlay  # noqa: E402

SIMS = 175


def ply_ms(sp, reps=3):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        sp.step()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def begin_cost(model, eng):
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for n in (4096, 7104):
        sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=n, max_iters=32, reuse_tree=True)
        for _ in range(8):
            sp.step()
        ms = ply_ms(sp)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                sp.step()
            torch.cuda.synchronize()
        k = {}
        for ev in prof.key_averages():
            for name in ("k_mcts_reuse_match", "k_mcts_reuse_gather", "k_mcts_reuse_commit"):
                if name in ev.key:
                    k[name] = k.get(name, 0.0) + ev.device_time_total / 3 / 1e3        # ms per ply
        s = sp.stats()
        out[str(n)] = dict(slots=n, ply_ms=ms, reuse_kernels_ms_per_ply=k, reuse_share_of_ply=sum(k.values()) / ms,
                           reused_searches=s["reused_searches"], fresh_searches=s["fresh_searches"])
        print("begin cost %d slots:" % n, out[str(n)], flush=True)
        del sp
    return out


def selfplay(model, eng):
    out = {}
    for n in (180, 4096):
        for rep in range(2):
            for reuse in (False, True):
                sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=n, max_iters=32, reuse_tree=reuse)
                for _ in range(7):
                    sp.step()
                ms = ply_ms(sp)
                key = "%d_%s" % (n, "reuse" if reuse else "fresh")
                out.setdefault(key, []).append(dict(ms_per_ply=ms, sims_per_s=n * SIMS / ms * 1e3))
                print("self-play %d slots reuse=%s: %.3f ms per ply" % (n, reuse, ms), flush=True)
                del sp
    return out


def carried(model, eng, n=1024, iters=60):
    sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=n, max_iters=128, reuse_tree=True)
    rows = []
    for it in range(iters):
        sp.step()
        r, v = sp.reused, sp.visits.sum(1)
        active = (r >= 0)
        carried_ = r > 0
        na, nc = int(active.sum()), int(carried_.sum())
        mean = float((v[carried_] - (SIMS + 1)).double().mean()) if nc else None
        rows.append(dict(iteration=it, active=na, carried=nc, share=nc / na if na else None, mean_carried_root_visits=mean))
    s = sp.stats()
    return dict(slots=n, by_iteration=rows, reused_searches=s["reused_searches"], fresh_searches=s["fresh_searches"])


def pool(model, eng):
    out = {}
    for reuse in (False, True):
        sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=4096, max_iters=16, reuse_tree=reuse)
        for _ in range(6):
            sp.step()
        torch.cuda.synchronize()
        out["reuse" if reuse else "fresh"] = int(eng.L.ccx_mcts_pool_bytes(eng.h))
        del sp
    return out


def match(a, b, ka, kb, games, seed):
    """a (BatchedArena side options ka) against b (kb), a moving first in the first half of the games, second in the other"""
    half = games // 2
    r1 = BatchedArena(a, b, half, seed=seed, enforce_move_limit=True, leaves_per_round=(ka[0], kb[0]), reuse_tree=(ka[1], kb[1])).play()
    r2 = BatchedArena(b, a, games - half, seed=seed, game_id0=half, enforce_move_limit=True, leaves_per_round=(kb[0], ka[0]),
                      reuse_tree=(kb[1], ka[1])).play()
    wins, losses = r1["p1_wins"] + r2["p2_wins"], r1["p2_wins"] + r2["p1_wins"]
    return dict(games=games, wins=wins, losses=losses, draws_or_unfinished=games - wins - losses,
                win_rate_of_decided=wins / (wins + losses) if wins + losses else None, wilson95=wilson(wins, wins + losses))


def strength(model, games, seed=2026):
    other = ResidualCNN(engine=Engine(0)).load_weights(WEIGHTS).set_kernel("tc_acc")
    t0 = time.perf_counter()
    reuse_vs_fresh = match(model, other, (1, True), (1, False), games, seed)
    print("L=1 reuse vs L=1 fresh:", reuse_vs_fresh, flush=True)
    l8_vs_l1 = match(model, other, (8, True), (1, False), games, seed + 1)
    print("L=8 reuse vs L=1 fresh:", l8_vs_l1, flush=True)
    return dict(l1_reuse_vs_l1=reuse_vs_fresh, l8_reuse_vs_l1=l8_vs_l1, seconds=time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--games", type=int, default=1024)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("reuse_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    eng = Engine(0)
    model = ResidualCNN(engine=eng).load_weights(WEIGHTS).set_kernel("tc_acc")
    res = dict(card=card(), simulations=SIMS, net_mode="tc_acc", carry=3)
    res["begin"] = begin_cost(model, eng)
    res["selfplay"] = selfplay(model, eng)
    res["carried"] = carried(model, eng)
    res["pool_bytes"] = pool(model, eng)
    res["strength"] = strength(model, args.games)
    res["card_after"] = card()
    path = os.path.join(args.out, "reuse_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
