"""Where the random-legal env step's warp time goes, counted on the CPU, and a model of the carry-over schedule.

Steps `--games` games from the start position with a host build of the kernels' own ply code (scripts/fill_count.cu over
ccx_device.cuh), skips `--warmup` plies and records the fill steps of every later game-ply.  Then, for warps of 32 games:
- the expansion histogram, the mean over lanes and the mean max over a warp's lanes per ply, whose ratio is the lane
  utilisation of k_step_random_pick's fill loop (the warp runs each ply's fill as long as its longest lane);
- issued warp instructions per 32 game-plies, modelled as `--fixed` per round in which any lane finishes or starts a ply
  plus `--fill` per fill iteration, for the lockstep kernel (k_step_random_pick) and for k_step_random_carry at each K
  (a round runs at most K fill steps per lane; a lane whose fill is done finishes and starts a ply in the next round).
  With `--peel` a ready lane takes the first fill step of the ply it starts inside the per-ply path (count it in `--fixed`),
  so the round's K steps begin at the ply's second.
The default costs are SASS counts of k_step_random_carry (DESIGN.md §3); redo them and the choice of K after changing it.  The
lockstep line uses the same costs, so it stands for the lockstep schedule of this ply code, not for k_step_random_pick as built.
The model ignores divergence, latency and registers, so it ranks schedules; only a GPU run times them.
usage: python scripts/fill_model.py [--games 8192] [--plies 5888] [--warmup 768] [--fixed 277] [--fill 34] [--peel]"""
import argparse
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def count(games, plies, warmup, seed):
    with tempfile.TemporaryDirectory() as tmp:
        lib = os.path.join(tmp, "libfill_count.so")
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        env = dict(os.environ)
        env.pop("CC", None)
        env.pop("CXX", None)
        subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                               "-shared", "-o", lib, os.path.join(HERE, "fill_count.cu")], env=env)
        L = ctypes.CDLL(lib)
        L.fc_count.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p]
        L.fc_count.restype = ctypes.c_longlong
        E = np.zeros((games, plies - warmup), dtype=np.uint8)
        nowalk = L.fc_count(games, plies, warmup, seed, E.ctypes.data)
    return E, nowalk


def lockstep_cost(E, fixed, fill):
    """k_step_random_pick: every ply costs the fixed path plus the warp's longest fill"""
    W = E.reshape(-1, 32, E.shape[1])
    return (fixed + fill * W.max(axis=1)).sum(axis=1).mean()


def carry_cost(E, K, fixed, fill, peel=False):
    """k_step_random_carry with at most K fill steps per lane and round (after the first, with `peel`); returns (cost, rounds)
    per warp"""
    W = E.reshape(-1, 32, E.shape[1]).astype(np.int64)
    nw, P = W.shape[0], W.shape[2]
    wi, li = np.meshgrid(np.arange(nw), np.arange(32), indexing="ij")
    ply = np.zeros((nw, 32), np.int64)
    rem = np.zeros((nw, 32), np.int64)
    pending = np.zeros((nw, 32), bool)             # a ply picked, its fill running or done
    cost = np.zeros(nw)
    rounds = np.zeros(nw)
    while True:
        ready = rem == 0
        fin = ready & pending                      # finish the ply
        ply += fin
        pending &= ~fin
        start = ready & (ply < P)
        while True:                                # start the next ply; a ply that passes (0 steps) is skipped in place
            r = np.where(start, W[wi, li, np.minimum(ply, P - 1)], 0)
            skip = start & (r == 0)
            if not skip.any():
                break
            ply += skip
            start &= ply < P
        rem = np.where(start, r - int(peel), rem)
        pending |= start
        path = (fin | start).any(axis=1)
        if not (path.any() or pending.any()):
            break
        steps = np.minimum(rem, K)
        cost += np.where(path, fixed, 0) + fill * steps.max(axis=1)
        rounds += path | pending.any(axis=1)
        rem -= steps
    return cost.mean(), rounds.mean()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--games", type=int, default=8192)
    ap.add_argument("--plies", type=int, default=5888, help="plies stepped, warm-up included")
    ap.add_argument("--warmup", type=int, default=768)
    ap.add_argument("--seed", type=lambda s: int(s, 0), default=0x5EED2026)
    ap.add_argument("--fixed", type=float, default=277.0, help="warp instructions of the per-ply path")
    ap.add_argument("--fill", type=float, default=34.0, help="warp instructions of one fill iteration")
    ap.add_argument("--k", type=int, nargs="+", default=[3, 4, 5, 6, 8])
    ap.add_argument("--peel", action="store_true", help="the ply start takes the fill's first step")
    a = ap.parse_args()
    assert a.games % 32 == 0 and a.plies > a.warmup
    E, nowalk = count(a.games, a.plies, a.warmup, a.seed)
    P = E.shape[1]
    gp = E.size
    print("%d games x %d plies after %d warm-up plies: %d game-plies" % (a.games, P, a.warmup, gp))
    h = np.bincount(E.ravel(), minlength=11)
    print("fill steps per game-ply: " + "  ".join("%d: %.1f %%" % (k, 100 * h[k] / gp) for k in range(10))
          + "  >=10: %.1f %%" % (100 * h[10:].sum() / gp))
    mean = E.mean()
    wmax = E.reshape(-1, 32, P).max(axis=1).mean()
    print("mean %.2f per game-ply, mean max over a warp's 32 lanes %.2f per ply: lane utilisation %.1f %%" % (mean, wmax, 100 * mean / wmax))
    print("walk-test expansions (checkers without an empty neighbour): %.4f per game-ply" % (nowalk / gp))
    base = lockstep_cost(E, a.fixed, a.fill)
    per32 = lambda c: c / P
    print("model: %.0f per round with a ply to finish or start, %.0f per fill iteration; warp instructions per 32 game-plies"
          % (a.fixed, a.fill))
    print("  lockstep (k_step_random_pick): %.0f  1.00x" % per32(base))
    for K in a.k:
        c, r = carry_cost(E, K, a.fixed, a.fill, a.peel)
        print("  carry K=%d%s: %.0f  %.2fx  (%.2f rounds per ply)" % (K, " (first step in the ply start)" if a.peel else "", per32(c),
                                                                     base / c, r / P))


if __name__ == "__main__":
    main()
