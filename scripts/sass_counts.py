"""SASS instruction counts of the carry env step's one-wave kernel, k_step_random_carry<false, 448, 1, 5>, and registers and
spills of all four carry instantiations.

Compiles chinesecheckersagent_b200/csrc/ccx_env.cu (or the file given) to a cubin with the library's flags and -Xptxas -v,
then reads the kernel's SASS (cuobjdump -sass):
- round path: the main loop's head (the target of its longest backward branch) up to the first fill step's first FLO.U32
  (a fill step takes the top bit of `todo` from two FLO.U32 a few instructions apart),
  every instruction in between counted once, so it holds the rare blocks too (win reset, no-walk expansions, pass);
- fill step: the first unrolled fill step, from its first FLO.U32 up to and including its exit branch;
- with --taken: the common round path, walked from the loop head to the first fill step, following the conditional
  branches whose addresses are listed (hex) and falling through the others.  The list is read off the SASS, for the round
  in which a lane finishes a ply without a win and starts the next with a walk for every checker.
Opcodes are split by pipe as scripts/pipe_rates.py measured them on B200: ALU (LOP3, SHF, ISETP, PRMT, SEL, IADD3, VIMNMX,
PLOP3, LEA, ...) and the IMAD pipe (IMAD in every form, VIADD); FLO / POPC / BREV, the loads and control flow are counted apart.
CPU only.
usage: python scripts/sass_counts.py [--taken 1d20,2590,...] [path/to/ccx_env.cu]"""
import argparse
import collections
import os
import re
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "..", "chinesecheckersagent_b200", "csrc", "ccx_env.cu")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--fmad=false"]
KERNEL = "_Z19k_step_random_carryILb0ELi448ELi1ELi5E"
IMAD_PIPE = {"IMAD", "VIADD"}
OTHER = {"FLO", "POPC", "BREV", "LDS", "LDG", "STG", "LDCU", "LDC", "S2UR", "S2R", "BRA", "BSSY", "BSYNC", "BREAK", "EXIT",
         "WARPSYNC", "UMOV", "ULEA", "UIADD3", "UISETP", "NOP", "ATOMG", "REDG", "RED"}


def compile_cubin(src, tmp):
    out = os.path.join(tmp, "env.cubin")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    res = subprocess.run([nvcc, "-cubin"] + FLAGS + ["-Xptxas", "-v", "-o", out, src], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, env=env, check=True)
    return out, res.stdout


def registers(ptxas):
    """{kernel template arguments: (registers, spill stores, spill loads)} of the carry kernels"""
    out, name = {}, None
    for line in ptxas.splitlines():
        m = re.search(r"entry function '_Z19k_step_random_carryILb(\d)ELi(\d+)ELi(\d)ELi(\d)E", line)
        if m:
            name = "<%s, %s, %s, %s>" % ("true" if m.group(1) == "1" else "false", m.group(2), m.group(3), m.group(4))
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            out.setdefault(name, [0, 0, 0])[1:] = [int(m.group(1)), int(m.group(2))]
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            out.setdefault(name, [0, 0, 0])[0] = int(m.group(1))
            name = None
    return out


def kernel_sass(cubin):
    """[(address, opcode, full text)] of KERNEL"""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    sass = subprocess.run([cuobjdump, "-sass", cubin], check=True, stdout=subprocess.PIPE, text=True).stdout
    ins, on = [], False
    for line in sass.splitlines():
        if "Function :" in line:
            on = KERNEL in line
            continue
        m = re.search(r"/\*([0-9a-f]{4,})\*/\s+((?:@!?U?P\w+\s+)?([A-Z0-9_]+)[^;]*);", line)
        if on and m:
            ins.append((int(m.group(1), 16), m.group(3), m.group(2).strip()))
    return ins


def target(text):
    m = re.search(r"BRA(?:\s+!?U?P\w+,)?\s+(?:`\(\.L_x_\d+\)|0x([0-9a-f]+))", text)
    return int(m.group(1), 16) if m and m.group(1) else None


def classes(ops):
    c = collections.Counter(ops)
    alu = sum(n for op, n in c.items() if op not in IMAD_PIPE and op not in OTHER)
    imad = sum(n for op, n in c.items() if op in IMAD_PIPE)
    return c, alu, imad


def report(title, ins):
    c, alu, imad = classes([op for _, op, _ in ins])
    print("%s: %d instructions, ALU pipe %d, IMAD pipe %d" % (title, len(ins), alu, imad))
    print("  " + ", ".join("%s %d" % kv for kv in c.most_common()))


def common_path(ins, head, stop, taken):
    at = {a: k for k, (a, _, _) in enumerate(ins)}
    k, out = at[head], []
    while k != stop:
        a, op, t = ins[k]
        out.append(ins[k])
        if op == "BRA" and (not t.startswith("@") or a in taken):
            k = at[target(t)]
        else:
            k += 1
        if len(out) > 5000:
            raise RuntimeError("the common path does not reach the fill step")
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("src", nargs="?", default=SRC)
    ap.add_argument("--taken", default="")
    args = ap.parse_args()
    taken = {int(x, 16) for x in args.taken.split(",") if x}
    with tempfile.TemporaryDirectory() as tmp:
        cubin, ptxas = compile_cubin(args.src, tmp)
        ins = kernel_sass(cubin)
    regs = registers(ptxas)
    print("# registers / spill stores / spill loads (ptxas -v): " + ", ".join(
        "%s %d / %d / %d" % (k, *v) for k, v in sorted(regs.items())))
    back = [(a, target(t)) for a, op, t in ins if op == "BRA" and target(t) is not None and target(t) < a]
    end, head = max(back, key=lambda x: x[0] - x[1])
    addr = [a for a, _, _ in ins]
    flo = [k for k, (a, op, t) in enumerate(ins) if a > head and op == "FLO" and not t.startswith("FLO.U32.SH")
           and any(o == "FLO" for _, o, _ in ins[k + 1:k + 4])]
    h = addr.index(head)
    report("round path, loop head to the first fill step", ins[h:flo[0]])
    if taken:
        report("common round path (taken: %s)" % ",".join("%x" % a for a in sorted(taken)), common_path(ins, head, flo[0], taken))
    k = flo[0]
    while ins[k][1] != "BRA":
        k += 1
    step = ins[flo[0]:k + 1]
    report("unrolled fill step, FLO to its exit branch", step)
    for _, _, t in step:
        print("   " + t)


if __name__ == "__main__":
    main()
