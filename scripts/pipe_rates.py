"""Sustained issue rate of single integer instruction classes on the GPU (scripts/pipe_rates.cu): LOP3, SHF, IADD3, PRMT,
VIMNMX, IMAD, FLO and POPC alone, and VIADD / IMAD.IADD / IMAD / IADD3 interleaved with a second class (ptxas folds a stream of
immediate adds and turns a stream of mad-by-one into IADD3).  One 1,024-lane block per SM (8 warps per scheduler), eight
independent chains per lane.

The SASS of every stream's loop (cuobjdump -sass of the built library, from the loop head to its backward branch) gives the
opcodes and their counts per iteration; the rate is warp instructions per scheduler per cycle (clock64 cycles of each block,
median over blocks; four schedulers per SM).  The card's name, power limit and max SM clock are printed first.
usage: python scripts/pipe_rates.py [--iters 4096]"""
import argparse
import collections
import ctypes
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
THREADS = 1024
SCHEDULERS = 4


def build(tmp):
    lib = os.path.join(tmp, "libpipe_rates.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-o", lib, os.path.join(HERE, "pipe_rates.cu")], env=env)
    return lib


def loop_opcodes(lib):
    """{stream name: Counter of the SASS opcodes (without modifiers) of its loop body}"""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    sass = subprocess.run([cuobjdump, "-sass", lib], check=True, stdout=subprocess.PIPE, text=True).stdout
    out, name, ins = {}, None, []

    def close():
        if name is None:
            return
        loops = [(t, k) for k, (a, op, t) in enumerate(ins) if op == "BRA" and t is not None and t < a]
        t, k = max(loops, key=lambda x: ins[x[1]][0] - x[0])            # the longest backward branch: the stream's loop
        out[name] = collections.Counter(op for a, op, _ in ins if t <= a <= ins[k][0] and op != "BRA")

    for line in sass.splitlines():
        m = re.search(r"Function : _Z\d+k_rate_(\w+?)ij", line)
        if m:
            close()
            name, ins = m.group(1), []
            continue
        m = re.search(r"/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_]+)[^;]*?(?:\s0x([0-9a-f]+))?\s*;", line)
        if m and name:
            ins.append((int(m.group(1), 16), m.group(2), int(m.group(3), 16) if m.group(2) == "BRA" and m.group(3) else None))
    close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--iters", type=int, default=4096)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    print("# %s (nvidia-smi name, power.limit, clocks.max.sm)" % (q[0] if q else "nvidia-smi unavailable"))
    torch.cuda.init()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    with tempfile.TemporaryDirectory() as tmp:
        lib = build(tmp)
        ops = loop_opcodes(lib)
        L = ctypes.CDLL(lib)
    L.pr_name.restype = ctypes.c_char_p
    L.pr_run.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    warps = THREADS // 32
    print("# %d SMs, one %d-lane block per SM (%d warps per scheduler), %d loop iterations" % (sms, THREADS, warps // SCHEDULERS,
                                                                                                args.iters))
    print("# stream: SASS opcodes per loop iteration -> warp instructions per scheduler-cycle, per opcode and in all")
    for k in range(L.pr_count()):
        name = L.pr_name(k).decode()
        cyc = np.zeros(sms, np.int64)
        ms = ctypes.c_float(0)
        rc = L.pr_run(k, sms, THREADS, args.iters, cyc.ctypes.data_as(ctypes.c_void_p), ctypes.byref(ms))
        if rc != 0:
            raise RuntimeError("pipe_rates: CUDA error %d in stream %s" % (rc, name))
        c = float(np.median(cyc))
        body = ops[name]
        per = {op: n * args.iters * warps / SCHEDULERS / c for op, n in body.most_common()}
        print("%-14s %-40s -> %s  all %.3f  (%.0f cycles, %.3f ms)" % (
            name, " ".join("%s x%d" % (op, n) for op, n in body.most_common()),
            " ".join("%s %.3f" % (op, r) for op, r in per.items()), sum(per.values()), c, ms.value))


if __name__ == "__main__":
    main()
