"""Self-play resignation (resign_threshold / ccx_selfplay_resign): threshold calibration, plies per game, wall time, records and
the measured false-positive rate with resignation off and on, and the per-ply cost of the check.

    python scripts/resign_bench.py --out DIR [--reps 3]

Writes DIR/r07_resign_bench.json with:
  calibration  one track-only run (threshold -1: never resigns, every won game leaves its winner's sample) of 8,192 games on
               4,096 slots: the suggested thresholds for false-positive targets 0.05 and 0.02
  games_180    play_games(180) on 180 slots (one evolve iteration at the reference's NUM_SELF_PLAY), resignation off against the
               f = 0.05 threshold with resign_probe 0.1, the two arms alternating `reps` times: wall time (host clock around the
               call, which ends in a device synchronise), mean / p95 / max plies per game, records kept
  games_8192   the same for play_games(8,192) on 4,096 slots, plus games/s and the probes' measured false-positive rate
  check_cost   torch.profiler (CUDA activities) over 4 plies of a 4,096-slot run with resignation on, in a run of its own:
               device time per ply of k_selfplay_resign and k_selfplay_resign_account against the ply's total kernel time
Every run uses the shipped net in the accurate mode and 175 simulations.  Plies per game are each ended game's ply count (the
opening's random plies included; a resigned game ends without a move).  The card's name, power limit and max SM clock are read by the same process."""
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
from chinesecheckersagent_b200.engine import Engine  # noqa: E402
from chinesecheckersagent_b200.model import ResidualCNN  # noqa: E402
from chinesecheckersagent_b200.selfplay import BatchedSelfPlay  # noqa: E402

WEIGHTS = os.path.join(ROOT, "tests", "golden", "good_model_weights.npz")
SIMS = 175


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


class GamePlies:
    """plies of every game that ends, read from its state just before ccx_selfplay_finish settles it (the ply count in META;
    a resigned game ends without a move); device tensors, no host sync per ply"""

    def __init__(self, sp):
        self.sp, self.rows, self.call = sp, [], sp.eng.call
        sp.eng.call = self._call

    def _call(self, name, *args):
        if name == "ccx_selfplay_finish":
            meta = self.sp.env.state[4]
            ended = ((meta >> 56) != 0) & (self.sp.start_iter <= self.sp.iter)
            self.rows.append(torch.where(ended, (meta >> 32) & 0xFFFF, -1))
        return self.call(name, *args)

    def close(self):
        self.sp.eng.call = self.call
        p = torch.cat(self.rows).cpu().numpy()
        return p[p >= 0].astype(np.float64)


def run(model, n, games, threshold, probe=0.1):
    kw = dict(resign_threshold=threshold, resign_probe=probe) if threshold is not None else {}
    sp = BatchedSelfPlay(model.eng, model.evaluate_states, n_slots=n, num_itr=SIMS, max_iters=512, seed=2026, **kw)
    gp = GamePlies(sp)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st = sp.play_games(games)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    plies = gp.close()
    out = dict(wall_s=wall, games_per_s=st["games_started"] / wall, plies_mean=float(plies.mean()), plies_p95=float(np.percentile(plies, 95)),
               plies_max=float(plies.max()), games_ended=int(plies.size), records=st["records"], kept_games=st["games"],
               discarded=st["discarded_repetition"] + st["discarded_no_progress"] + st["discarded_overflow"], plies=st["plies"],
               iterations=st["iterations"])
    if threshold is not None:
        out.update({k: st[k] for k in ("resigned_games", "probe_games", "probe_would_resign", "probe_false_positives",
                                       "false_positive_rate")})
    return out, sp


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    eng = Engine(0)
    model = ResidualCNN(engine=eng).load_weights(WEIGHTS)
    model.set_kernel("tc_acc")
    res = dict(card=card(), sims=SIMS, net="tests/golden/good_model_weights.npz, accurate mode")
    cal, sp = run(model, 4096, 8192, -1.0)
    res["calibration"] = dict(cal, samples=int(sp.resign_samples().size), threshold_f05=sp.suggest_resign_threshold(0.05),
                              threshold_f02=sp.suggest_resign_threshold(0.02))
    t05 = res["calibration"]["threshold_f05"]
    print("calibration", res["calibration"], flush=True)
    for key, n, games in (("games_180", 180, 180), ("games_8192", 4096, 8192)):
        arms = {"off": [], "on": []}
        for _ in range(a.reps):
            for arm, thr in (("off", None), ("on", t05)):
                r, _ = run(model, n, games, thr)
                arms[arm].append(r)
                print(key, arm, r, flush=True)
        res[key] = dict(threshold=t05, resign_probe=0.1, **arms)
    from torch.profiler import ProfilerActivity, profile
    sp = BatchedSelfPlay(eng, model.evaluate_states, n_slots=4096, num_itr=SIMS, max_iters=64, seed=7, resign_threshold=t05)
    for _ in range(10):
        sp.step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(4):
            sp.step()
        torch.cuda.synchronize()
    us = {}
    total = 0.0
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if ev.key.startswith(("k_", "void k_", "_Z")) or "k_" in ev.key:
            total += t
        if "resign" in ev.key:
            us[ev.key] = t / 4
    res["check_cost"] = dict(slots=4096, per_ply_us=us, ply_kernel_us=total / 4)
    print("check_cost", res["check_cost"], flush=True)
    with open(os.path.join(a.out, "r07_resign_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
