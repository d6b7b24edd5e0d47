"""A/B of the env step kernels (CCX_STEP_VARIANT): 10 = k_step_random_pick (default) against 9 = k_step_random_wq, the
all-six-closures kernel it replaced.  Bit-identity of state and win counters, and timing: 256-ply launches with the L2
flushed in between, the two arms alternated launch by launch at each size so that both see the same clocks and neighbours.
usage: python scripts/env_variants.py [games ...]"""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from chinesecheckersagent_b200.engine import BatchedEnv, Engine

eng = Engine(0)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
sizes = [int(x) for x in sys.argv[1:]] or [65536, 1048576]
ARMS = ("10", "9")
REPS = 7


def step(env, variant):
    os.environ["CCX_STEP_VARIANT"] = variant
    env.step_random(256)


for n in sizes:
    envs = {v: BatchedEnv(n, engine=eng, seed=0x5EED2026) for v in ARMS}
    for v in ARMS:                                   # first launch: compared below; two more to warm up
        step(envs[v], v)
    same = bool(torch.equal(envs["10"].state[:5], envs["9"].state[:5]) and torch.equal(envs["10"].wins, envs["9"].wins))
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
    for v, name in (("9", "k_step_random_wq (reference)"), ("10", "k_step_random_pick (default)")):
        m = ms[v][REPS // 2]
        print("n=%d variant %s %s: median %.3f ms (min %.3f, max %.3f)  %.3e steps/s" % (n, v, name, m, ms[v][0], ms[v][-1], n * 256 / m * 1e3), flush=True)
    print("n=%d speedup %.2fx  identical=%s" % (n, ms["9"][REPS // 2] / ms["10"][REPS // 2], same), flush=True)
os.environ.pop("CCX_STEP_VARIANT", None)
