"""ctypes binding of the tree-reuse oracle (reuse_oracle.c) — TEST INFRASTRUCTURE, NOT PRODUCT.

The library is built with gcc from reuse_oracle.c (which includes the leaf-parallel oracle, tests/leaves_oracle/leaves_oracle.c)
plus the one-leaf oracle's sources (oracle/ccx_oracle*.c) and lives next to this file (git-ignored)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ORACLE = os.path.join(ROOT, "oracle")
LEAVES = os.path.join(ROOT, "tests", "leaves_oracle", "leaves_oracle.c")
LIB = os.path.join(HERE, "libreuse_oracle.so")
NACT = 294
EVAL_UNIFORM, EVAL_HASH = 0, 1


def _sources():
    return [os.path.join(HERE, "reuse_oracle.c")] + sorted(
        os.path.join(ORACLE, f) for f in os.listdir(ORACLE) if f.startswith("ccx_oracle") and f.endswith(".c"))


def build():
    srcs = _sources()
    deps = srcs + [LEAVES, os.path.join(ORACLE, "ccx_oracle.h")]
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
        sig = {
            "rvo_forest_new": (vp, []),
            "rvo_forest_free": (None, [vp]),
            "rvo_forest_invalidate": (None, [vp]),
            "rvo_forest_begin": (None, [vp, vp, i64, i32, i32, i32, i32, i32, vp, vp, i32, i32, vp]),
            "rvo_forest_search": (None, [vp, i32, i32, dbl, i32, vp, i32, i32, i32, u64, i64, i32]),
            "rvo_forest_finalize": (None, [vp, dbl, vp, vp, vp, vp, vp, vp, vp]),
            "rvo_forest_child_stats": (None, [vp, i64, i32, vp, vp, vp]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


class Forest:
    """Persistent trees of the reuse begin (include/ccx.h ccx_mcts_begin_reuse), one per root, across searches:
    begin (re-root by state match under the carry rule, or fresh), search (`sims` selections per active tree in rounds of up
    to `leaves`), finalize.  S = the begin's num_itr, as the engine's search_with passes it (simulations + 1)."""

    def __init__(self):
        self.L = lib()
        self.f = self.L.rvo_forest_new()
        self.n = 0

    def __del__(self):
        if getattr(self, "f", None):
            self.L.rvo_forest_free(self.f)
            self.f = None

    def invalidate(self):
        """a new evaluator: the next begin starts every tree fresh"""
        self.L.rvo_forest_invalidate(self.f)

    def begin(self, st, S, carry, prev=None, noise=None, normalize=0, min_ply=-1, ply_parity=-1, edges_per_tree=0):
        st = np.ascontiguousarray(st, dtype=np.uint64)
        n = st.shape[1]
        prev = None if prev is None else np.ascontiguousarray(prev, dtype=np.int64)
        noise = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64)
        reused = np.zeros(n, dtype=np.int32)
        self.L.rvo_forest_begin(self.f, _ptr(st), n, S, edges_per_tree, min_ply, ply_parity, carry, _ptr(prev), _ptr(noise),
                                0 if noise is None else noise.shape[1], normalize, _ptr(reused))
        self.n = n
        return reused

    def search(self, sims, leaves=1, cpuct=3.5, evaluator=EVAL_UNIFORM, noise=None, normalize=0, ties=None, nthreads=8):
        """noise: mixed into a root when this search expands it"""
        noise = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64)
        seed, uid0 = ties if ties is not None else (0, 0)
        self.L.rvo_forest_search(self.f, sims, leaves, cpuct, evaluator, _ptr(noise), 0 if noise is None else noise.shape[1],
                                 normalize, int(ties is not None), int(seed), int(uid0), nthreads)

    def finalize(self, tau=1.0, stats=None):
        """(visits, pi, root Q, node count) as the engine's finalize; a dict `stats` receives vl_left, root W and P"""
        n = self.n
        visits = np.zeros((n, NACT), dtype=np.uint32)
        pi, q, W, P = (np.zeros((n, NACT), dtype=np.float64) for _ in range(4))
        nodes = np.zeros(n, dtype=np.int32)
        vl = np.zeros(n, dtype=np.int64)
        self.L.rvo_forest_finalize(self.f, tau, _ptr(visits), _ptr(pi), _ptr(q), _ptr(nodes), _ptr(vl), _ptr(W), _ptr(P))
        if stats is not None:
            stats.update(vl_left=vl, W=W, P=P)
        return visits, pi, q, nodes

    def child_stats(self, i, act):
        """(N, W, P) by policy index of the root edges of tree i's child along policy index `act`"""
        N = np.zeros(NACT, dtype=np.uint32)
        W, P = np.zeros(NACT), np.zeros(NACT)
        self.L.rvo_forest_child_stats(self.f, int(i), int(act), _ptr(N), _ptr(W), _ptr(P))
        return N, W, P
