"""A/B of the env step kernels (CCX_STEP_VARIANT): 11 = k_step_random_carry (default) against 10 = k_step_random_pick, the
lockstep kernel it replaced, and 9 = k_step_random_wq, the all-six-closures kernel before that.  Bit-identity of state and
win counters, and timing: 256-ply launches with the L2 flushed in between, the arms alternated launch by launch at each size
so that all see the same clocks and neighbours.
usage: python scripts/env_variants.py [games ...]"""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from chinesecheckersagent_b200.engine import BatchedEnv, Engine

eng = Engine(0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
sizes = [int(x) for x in sys.argv[1:]] or [65536, 1048576]
ARMS = ("11", "10", "9")
NAMES = {"11": "k_step_random_carry (default)", "10": "k_step_random_pick", "9": "k_step_random_wq"}
REPS = 7


def step(env, variant):
    os.environ["CCX_STEP_VARIANT"] = variant
    env.step_random(256)


for n in sizes:
    envs = {v: BatchedEnv(n, engine=eng, seed=0x5EED2026) for v in ARMS}
    for v in ARMS:                                   # first launch: compared below; two more to warm up
        step(envs[v], v)
    same = all(torch.equal(envs[v].state[:5], envs["9"].state[:5]) and torch.equal(envs[v].wins, envs["9"].wins) for v in ARMS)
    for _ in range(2):
        for v in ARMS:
            step(envs[v], v)
    ts = {v: [] for v in ARMS}
    for _ in range(REPS):
        for v in ARMS:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            flush.fill_(1); a.record(); step(envs[v], v); b.record(); ts[v].append((a, b))
    torch.cuda.synchronize()
    ms = {v: sorted(a.elapsed_time(b) for a, b in ts[v]) for v in ARMS}
    for v in reversed(ARMS):
        m = ms[v][REPS // 2]
        print("n=%d variant %s %s: median %.3f ms (min %.3f, max %.3f)  %.3e steps/s" % (n, v, NAMES[v], m, ms[v][0], ms[v][-1], n * 256 / m * 1e3), flush=True)
    print("n=%d speedup 11 over 10 %.3fx, over 9 %.2fx  identical=%s" % (n, ms["10"][REPS // 2] / ms["11"][REPS // 2],
                                                                        ms["9"][REPS // 2] / ms["11"][REPS // 2], same), flush=True)
os.environ.pop("CCX_STEP_VARIANT", None)
