"""Self-play playout cap randomization (full_search_prob / ccx_selfplay_playout_cap, budgets of ccx_mcts_begin_budget): ply time,
games, records and net rows with the cap off and on, and the default path against the parent build.

    python scripts/playout_cap_bench.py --out DIR [--reps 3] [--parent-root DIR]

Writes DIR/r09_playout_cap_bench.json with:
  ply_ms       per slot count (180, 4,096): device time per self-play ply (CUDA events around 8 steps after 12 warm-up steps, the
               warm-up covering the graph capture) for three arms alternating `reps` times: cap off; cap on (p = 0.25,
               fast_itr = 32); all budgets full (p = 1: the budgeted kernels doing the full work, against the cap-off path)
  games_8192   play_games(8,192) on 4,096 slots, cap off against cap on, alternating `reps` times: wall time (host clock around
               the call, which ends in a device synchronise), games/s, plies per game, records kept, full / fast searches
  net_rows     net rows per searched ply, computed on the host from the run's full / fast counts: every round's rows without
               compaction against the at most one row per selection of the compacted batch
  split        torch.profiler (CUDA activities) over 4 cap-on plies at 4,096 slots, in a run of its own: device time per ply of
               the tree kernels, the trunk and the policy dense kernel
  parent       with --parent-root (a directory holding the parent commit's package, library built): cap-off ply time of the
               parent against this tree, PUCT / symmetry off and PUCT / symmetry mean at 4,096 and 180 slots, alternating in child
               processes
Every run uses the shipped net in the accurate mode and 175 full simulations.  The card's name, power limit and max SM clock
are read by the same process."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WEIGHTS = os.path.join(ROOT, "tests", "golden", "good_model_weights.npz")
SIMS, FAST, P = 175, 32, 0.25


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def load():
    from chinesecheckersagent_b200.engine import Engine
    from chinesecheckersagent_b200.model import ResidualCNN
    eng = Engine(0)
    model = ResidualCNN(engine=eng).load_weights(WEIGHTS)
    model.set_kernel("tc_acc")
    return eng, model


def ply_ms(model, n, warm=12, steps=8, **kw):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=n, num_itr=SIMS, max_iters=64, seed=7, ring=True, **kw)
    for _ in range(warm):
        sp.step()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(steps):
        sp.step()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def games(model, cap):
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    kw = dict(full_search_prob=P, fast_itr=FAST) if cap else {}
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=4096, num_itr=SIMS, max_iters=512, seed=2026, **kw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st = sp.play_games(8192)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    out = dict(wall_s=wall, games_per_s=st["games_started"] / wall, plies=st["plies"], kept_games=st["games"], records=st["records"],
               plies_per_kept_game=st["plies"] / max(st["games"], 1), iterations=st["iterations"])
    if cap:
        out.update(full_searches=st["full_searches"], fast_searches=st["fast_searches"])
    return out


def child(args):
    """one cap-off ply-time measurement with the package under args.child_root (parent comparison)"""
    sys.path.insert(0, os.path.abspath(args.child_root))
    eng, model = load()
    n, sym = args.child_n, args.child_sym
    if sym != "off":
        model.set_symmetry(sym, 5)
    print(json.dumps(dict(ms=ply_ms(model, n))), flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent-root")
    ap.add_argument("--child-n", type=int)
    ap.add_argument("--child-sym")
    ap.add_argument("--child-root", default=ROOT)
    a = ap.parse_args()
    if a.child_n:
        return child(a)
    os.makedirs(a.out, exist_ok=True)
    eng, model = load()
    res = dict(card=card(), sims=SIMS, fast_itr=FAST, full_search_prob=P, net="tests/golden/good_model_weights.npz, accurate mode")
    arms = (("off", {}), ("cap", dict(full_search_prob=P, fast_itr=FAST)), ("all_full", dict(full_search_prob=1.0, fast_itr=FAST)))
    res["ply_ms"] = {}
    for n in (180, 4096):
        r = {k: [] for k, _ in arms}
        for _ in range(a.reps):
            for k, kw in arms:
                r[k].append(ply_ms(model, n, **kw))
        res["ply_ms"][str(n)] = r
        print("ply_ms", n, r, flush=True)
    g = {"off": [], "cap": []}
    for _ in range(a.reps):
        for k in g:
            g[k].append(games(model, k == "cap"))
            print("games_8192", k, g[k][-1], flush=True)
    res["games_8192"] = g
    full = sum(x["full_searches"] for x in g["cap"])
    fast = sum(x["fast_searches"] for x in g["cap"])
    rounds = SIMS + 1
    need = (full * (SIMS + 1) + fast * (FAST + 1)) / max(full + fast, 1)
    res["net_rows"] = dict(uncompacted_per_searched_ply=rounds, compacted_at_most_per_searched_ply=need, full_share=full / max(full + fast, 1),
                           note="rows per searched ply of one slot, from the budgets: without compaction every round evaluates every "
                                "slot's row; the compacted batch evaluates at most one row per selection (none for a terminal leaf)")
    print("net_rows", res["net_rows"], flush=True)
    from chinesecheckersagent_b200.selfplay import BatchedSelfPlay
    from torch.profiler import ProfilerActivity, profile
    sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=4096, num_itr=SIMS, max_iters=64, seed=7, full_search_prob=P, fast_itr=FAST)
    for _ in range(12):
        sp.step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(4):
            sp.step()
        torch.cuda.synchronize()
    split = {"tree": 0.0, "trunk": 0.0, "policy_dense": 0.0, "other": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        k = ev.key
        if "k_mcts" in k:
            split["tree"] += t
        elif "trunk" in k:
            split["trunk"] += t
        elif "policy_dense" in k:
            split["policy_dense"] += t
        elif "k_" in k:
            split["other"] += t
    res["split_us_per_ply"] = {k: v / 4 for k, v in split.items()}
    print("split", res["split_us_per_ply"], flush=True)
    eng.close()
    if a.parent_root:
        par = {}
        for sym in ("off", "mean"):
            for n in (4096, 180):
                r = {"parent": [], "this": []}
                for _ in range(a.reps):
                    for k in r:
                        root = a.parent_root if k == "parent" else ROOT
                        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-n", str(n), "--child-sym", sym,
                                              "--child-root", root], stdout=subprocess.PIPE, text=True, check=True).stdout
                        r[k].append(json.loads(out.strip().splitlines()[-1])["ms"])
                par["%s_%d" % (sym, n)] = r
                print("parent", sym, n, r, flush=True)
        res["parent"] = par
    with open(os.path.join(a.out, "r09_playout_cap_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
