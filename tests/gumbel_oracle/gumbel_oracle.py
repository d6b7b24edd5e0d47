"""ctypes binding of the Gumbel-search oracle (gumbel_oracle.c) — TEST INFRASTRUCTURE, NOT PRODUCT.

The library is built with gcc from gumbel_oracle.c plus the one-leaf oracle's sources (oracle/ccx_oracle*.c: board, encoding,
Philox, thread pool), including the kernels' csrc/ccx_fpmath.cuh and csrc/ccx_gumbel_table.h, and lives next to this file
(git-ignored)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ORACLE = os.path.join(ROOT, "oracle")
CSRC = os.path.join(ROOT, "chinesecheckersagent_b200", "csrc")
LIB = os.path.join(HERE, "libgumbel_oracle.so")
NACT = 294
EVAL_UNIFORM, EVAL_HASH = 0, 1


def _sources():
    return [os.path.join(HERE, "gumbel_oracle.c")] + sorted(
        os.path.join(ORACLE, f) for f in os.listdir(ORACLE) if f.startswith("ccx_oracle") and f.endswith(".c"))


def build():
    srcs = _sources()
    deps = srcs + [os.path.join(ORACLE, "ccx_oracle.h"), os.path.join(CSRC, "ccx_fpmath.cuh"), os.path.join(CSRC, "ccx_gumbel_table.h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in deps):
        return LIB
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-ffp-contract=off", "-shared", "-I", ORACLE,
                           "-I", CSRC, "-x", "c", "-o", LIB] + srcs + ["-lm", "-lpthread"])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        i64, i32, u64, dbl, vp = ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64, ctypes.c_double, ctypes.c_void_p
        L.gmo_mcts_batch.argtypes = [vp, i64, i32, i32, i32, dbl, dbl, dbl, u64, i64, vp, vp, vp, vp, vp, vp, vp, i32]
        L.gmo_mcts_batch.restype = None
        L.gmo_eval_batch.argtypes = [vp, i64, i32, vp, vp]
        L.gmo_eval_batch.restype = None
        L.gmo_log.argtypes = [dbl]
        L.gmo_log.restype = dbl
        L.gmo_exp.argtypes = [dbl]
        L.gmo_exp.restype = dbl
        L.gmo_considered_visits.argtypes = [i32, i32, vp]
        L.gmo_considered_visits.restype = None
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def mcts(st, num_itr=175, pre_expand=0, evaluator=EVAL_UNIFORM, considered=16, scale=1.0, c_visit=50.0, c_scale=0.1, seed=0,
         uid0=0, uids=None, nthreads=1):
    """The Gumbel search of BatchedMCTS(gumbel=True, num_itr, gumbel_*) with tie_uid0 = uid0 (or slot ids `uids`) on roots st
    (8, n).  Returns dict(visits u32, pi f64, q f64 (n, 294), action i32, n_nodes i32, in_considered i32 (n,))."""
    st = np.ascontiguousarray(st, dtype=np.uint64)
    n = st.shape[1]
    out = dict(visits=np.zeros((n, NACT), dtype=np.uint32), pi=np.zeros((n, NACT)), q=np.zeros((n, NACT)),
               action=np.zeros(n, dtype=np.int32), n_nodes=np.zeros(n, dtype=np.int32), in_considered=np.zeros(n, dtype=np.int32))
    if uids is not None:
        uids = np.ascontiguousarray(uids, dtype=np.int64)
    lib().gmo_mcts_batch(_ptr(st), n, int(num_itr) + int(bool(pre_expand)), evaluator, int(considered), float(scale), float(c_visit),
                         float(c_scale), int(seed) & 0xFFFFFFFFFFFFFFFF, int(uid0), _ptr(uids), _ptr(out["visits"]), _ptr(out["pi"]),
                         _ptr(out["q"]), _ptr(out["action"]), _ptr(out["n_nodes"]), _ptr(out["in_considered"]), nthreads)
    return out


def eval_batch(planes, evaluator=EVAL_HASH):
    planes = np.ascontiguousarray(planes, dtype=np.uint8)
    n = planes.shape[0]
    p = np.zeros((n, NACT))
    v = np.zeros(n)
    lib().gmo_eval_batch(_ptr(planes), n, evaluator, _ptr(p), _ptr(v))
    return p, v


def fm_log(x):
    return lib().gmo_log(float(x))


def fm_exp(x):
    return lib().gmo_exp(float(x))


def considered_visits(m, sims):
    out = np.zeros(max(sims, 1), dtype=np.int32)
    lib().gmo_considered_visits(int(m), int(sims), _ptr(out))
    return out[:sims]
