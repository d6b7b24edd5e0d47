"""Microbenchmark of the jump flood fill alone (scripts/fill_latency.cu): the fill k_step_random_carry ran before its per-cell
constants were computed with ALU instructions (old: FLO + a tri_cell_info load per step) against the one it runs now (new:
ALU constants, the first step taken in the ply start), at 14 and 28 warps per SM (one and two 448-lane blocks).

Fill start states come from the host model of the random-legal ply (`--games` games from the start position, the plies
after `--warmup`).  Every lane runs `--fills` fills in lockstep with its warp.  Printed per arm and size: ms per launch (CUDA
events, median of `--reps` launches, arms alternated launch by launch), and clock64 cycles per warp per fill step (the loop's
cycles over the warp's fill iterations, each iteration as long as its longest lane), averaged over warps; the two arms'
destination sets are compared.
usage: python scripts/fill_latency.py [--games 4096] [--plies 1024] [--warmup 768] [--fills 256] [--reps 9]"""
import argparse
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TPB = 448


def build(tmp):
    lib = os.path.join(tmp, "libfill_latency.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-o", lib, os.path.join(HERE, "fill_latency.cu")], env=env)
    L = ctypes.CDLL(lib)
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    L.fl_table_bytes.argtypes = []
    L.fl_table_bytes.restype = i64
    L.fl_table.argtypes = [vp]
    L.fl_table.restype = None
    L.fl_record.argtypes = [ci, ci, ci, ctypes.c_uint64, vp, i64]
    L.fl_record.restype = i64
    L.fl_run.argtypes = [ci, ci, vp, i64, ci, vp, vp, vp, vp]
    L.fl_run.restype = ci
    return L


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--plies", type=int, default=1024, help="plies stepped, warm-up included")
    ap.add_argument("--warmup", type=int, default=768)
    ap.add_argument("--seed", type=lambda s: int(s, 0), default=0x5EED2026)
    ap.add_argument("--fills", type=int, default=256, help="fills per lane and launch")
    ap.add_argument("--reps", type=int, default=9)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "fill_latency.py needs a GPU"
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    with tempfile.TemporaryDirectory() as tmp:
        L = build(tmp)
        cap = a.games * (a.plies - a.warmup)
        st = np.zeros((4, cap), np.uint64)
        n = L.fl_record(a.games, a.plies, a.warmup, a.seed, st.ctypes.data, cap)
        assert n > 2 * sms * TPB, n
        st = np.ascontiguousarray(st[:, :n])
        T3 = np.zeros(L.fl_table_bytes(), np.uint8)
        L.fl_table(T3.ctypes.data)
        dst = torch.from_numpy(st.view(np.int64)).cuda()
        dT3 = torch.from_numpy(T3).cuda()
        print("%d fill start states from %d games (plies %d..%d); %d fills per lane" % (n, a.games, a.warmup, a.plies - 1, a.fills))
        for bps in (1, 2):
            blocks = sms * bps
            lanes = blocks * TPB
            out = {}
            for arm in (0, 1):
                out[arm] = (torch.zeros(lanes // 32, dtype=torch.int64, device="cuda"), torch.zeros(lanes // 32, dtype=torch.int32, device="cuda"),
                            torch.zeros(lanes, dtype=torch.int64, device="cuda"))
            run = lambda arm: L.fl_run(arm, blocks, dst.data_ptr(), n, a.fills, dT3.data_ptr(), *(t.data_ptr() for t in out[arm]))
            for arm in (0, 1):                       # warm-up
                assert run(arm) == 0
            torch.cuda.synchronize()
            same = torch.equal(out[0][2], out[1][2])
            ts = {0: [], 1: []}
            cyc = {0: [], 1: []}
            for _ in range(a.reps):
                for arm in (0, 1):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); run(arm); e1.record()
                    ts[arm].append((e0, e1))
                    torch.cuda.synchronize()
                    c, it, _ = out[arm]
                    cyc[arm].append(float((c.double() / it.double()).mean()))
            for arm, name in ((0, "old (FLO + tri_cell_info load)"), (1, "new (ALU constants, first step in the start)")):
                ms = sorted(e0.elapsed_time(e1) for e0, e1 in ts[arm])
                cy = sorted(cyc[arm])
                print("%2d warps/SM  %-46s  %.3f ms (min %.3f, max %.3f)  %.1f cycles per warp fill step (min %.1f, max %.1f)"
                      % (14 * bps, name, ms[a.reps // 2], ms[0], ms[-1], cy[a.reps // 2], cy[0], cy[-1]), flush=True)
            it = out[0][1].double().sum().item() / (lanes // 32) / a.fills
            print("%2d warps/SM  %.2f fill iterations per warp and fill (lockstep); destination sets identical=%s" % (14 * bps, it, same), flush=True)


if __name__ == "__main__":
    main()
