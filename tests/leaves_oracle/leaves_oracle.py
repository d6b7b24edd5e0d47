"""ctypes binding of the leaf-parallel MCTS oracle (leaves_oracle.c) — TEST INFRASTRUCTURE, NOT PRODUCT.

The library is built with gcc from leaves_oracle.c plus the one-leaf oracle's sources (oracle/ccx_oracle*.c: board, encoding,
Philox, thread pool) and lives next to this file (git-ignored)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ORACLE = os.path.join(ROOT, "oracle")
LIB = os.path.join(HERE, "libleaves_oracle.so")
NACT = 294
EVAL_UNIFORM, EVAL_HASH = 0, 1


def _sources():
    return [os.path.join(HERE, "leaves_oracle.c")] + sorted(
        os.path.join(ORACLE, f) for f in os.listdir(ORACLE) if f.startswith("ccx_oracle") and f.endswith(".c"))


def build():
    srcs = _sources()
    deps = srcs + [os.path.join(ORACLE, "ccx_oracle.h")]
    if os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(s) for s in deps):
        return LIB
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-ffp-contract=off", "-shared", "-I", ORACLE,
                           "-o", LIB] + srcs + ["-lm", "-lpthread"])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(build())
        i64, i32, u64, dbl, vp = ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64, ctypes.c_double, ctypes.c_void_p
        L.lvo_mcts_batch.argtypes = [vp, i64, i32, dbl, dbl, i32, i32, vp, i32, vp, vp, vp, vp, i32, i32, u64, i64, i32, vp, vp]
        L.lvo_mcts_batch.restype = None
        L.lvo_eval_batch.argtypes = [vp, i64, i32, vp, vp]
        L.lvo_eval_batch.restype = None
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def mcts(st, num_itr=175, cpuct=3.5, tau=1.0, pre_expand=0, evaluator=EVAL_UNIFORM, noise=None, nthreads=1, ties=None, leaves=1,
         stats=None):
    """oracle.mcts with `leaves` (1..16) selections per tree per round under virtual loss.  ties=None: first maximal edge;
    ties=(seed, uid0): the engine's tie rule 1.  A dict passed as `stats` receives per-root arrays "visited" (nodes reached by
    a selection, root included) and "vl_left" (virtual losses left after the search).
    Returns (visits[n,294] u32, pi[n,294] f64, root Q[n,294] f64, node count[n])."""
    st = np.ascontiguousarray(st, dtype=np.uint64)
    n = st.shape[1]
    visits = np.zeros((n, NACT), dtype=np.uint32)
    pi = np.zeros((n, NACT), dtype=np.float64)
    q = np.zeros((n, NACT), dtype=np.float64)
    nodes = np.zeros(n, dtype=np.int32)
    visited = np.zeros(n, dtype=np.int32)
    vl_left = np.zeros(n, dtype=np.int64)
    stride = 0
    if noise is not None:
        noise = np.ascontiguousarray(noise, dtype=np.float64)
        stride = noise.shape[1]
    seed, uid0 = ties if ties is not None else (0, 0)
    lib().lvo_mcts_batch(_ptr(st), n, num_itr, cpuct, tau, pre_expand, evaluator, _ptr(noise), stride, _ptr(visits), _ptr(pi),
                         _ptr(nodes), _ptr(q), nthreads, int(ties is not None), int(seed), int(uid0), int(leaves), _ptr(visited),
                         _ptr(vl_left))
    if stats is not None:
        stats.update(visited=visited, vl_left=vl_left)
    return visits, pi, q, nodes


def eval_batch(planes, evaluator=EVAL_HASH):
    """The oracle's test evaluators on encoded positions: planes uint8 (n, 7, 7, 7) -> (p (n, 294) f64, v (n,) f64)."""
    planes = np.ascontiguousarray(planes, dtype=np.uint8)
    n = planes.shape[0]
    p = np.zeros((n, NACT), dtype=np.float64)
    v = np.zeros(n, dtype=np.float64)
    lib().lvo_eval_batch(_ptr(planes), n, evaluator, _ptr(p), _ptr(v))
    return p, v
