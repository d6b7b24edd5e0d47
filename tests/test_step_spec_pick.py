"""The carry-over env step's speculative ply start (carry_ply_start): the checker is picked as if every checker had a walk and
the fill is started at once; only a position with a checker without a walk runs the exact pick.  A host build of the
kernel's source checks every ply start of seeded random play, of crowded positions (checkers without a walk, some that cannot
move) and of near-win positions (wins and resets) against the exact pick and against pick_first_start: same checker,
same origin, same fill start and the same destination set.  No position of six checkers a side leaves the mover without a
move (test_no_pass_with_six_opponents), so the pass is checked on constructed boards whose other cells are filled.  The whole carry loop against the oracle is
test_step_carry_ply.py's.  CPU only: nvcc builds the kernel's source for the host."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle as orc
from test_step_pick_first import near_win_states

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "spec_pick.cu")
SEED = 0x5EED2026


@pytest.fixture(scope="module")
def sp(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("spec_pick") / "libspec_pick.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-cudart", "none", "-o", lib, SRC], env=env)
    L = ctypes.CDLL(lib)
    L.sp_check.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int,
                           ctypes.c_int, ctypes.c_void_p]
    L.sp_check.restype = None
    L.sp_check_boards.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int64, ctypes.c_int, ctypes.c_void_p]
    L.sp_check_boards.restype = None
    L.sp_boxed_in_count.argtypes = [ctypes.c_int]
    L.sp_boxed_in_count.restype = ctypes.c_int64
    return L


def check(sp, st, step0, plies, gid0, wide):
    st = np.array(st, dtype=np.uint64, order="C")
    out = np.zeros(5, dtype=np.int64)
    sp.sp_check(st.ctypes.data_as(ctypes.c_void_p), st.shape[1], gid0, SEED, step0, plies, wide,
                out.ctypes.data_as(ctypes.c_void_p))
    return report(out)


def report(out):
    bad, starts, fallback, passes, stuck = (int(x) for x in out)
    print("%d ply starts, fallback %d (%.3f %%), with a checker that cannot move %d, passes %d" % (
        starts, fallback, 100.0 * fallback / starts, stuck, passes))
    return bad, starts, fallback, passes, stuck


@pytest.mark.parametrize("wide", [1, 0], ids=["wide", "tri"])
def test_spec_pick_random_play(sp, wide):
    """about 10^6 ply starts of random play from the start position (won games restart)"""
    bad, starts, fallback, _, stuck = check(sp, orc.start_states(4096), 11, 256, 900, wide)
    assert starts == 4096 * 256
    assert bad == 0
    assert 0 < fallback < starts // 20         # rare (most of it in the opening, where the back checkers are boxed in)
    assert stuck > 0


@pytest.mark.parametrize("wide", [1, 0], ids=["wide", "tri"])
@pytest.mark.parametrize("kind", ["crowded", "near_win"])
def test_spec_pick_rare_positions(sp, kind, wide):
    if kind == "crowded":                      # Board(randomised=True) placements: checkers boxed in
        st, plies = orc.random_states(6000, seed=41), 40
    else:
        st, plies = near_win_states(3000, seed=43), 60
    bad, starts, fallback, passes, stuck = check(sp, st, 3, plies, 7000, wide)
    assert bad == 0
    assert fallback > 0
    assert stuck > 0


def boxed_boards(n, seed):
    """the mover's six checkers on random cells, the opponent on every other cell but 0-8 random empty ones: passes (no
    empty cell at all, or none the mover can reach), positions where some checkers cannot move, and plain fallbacks"""
    rng = np.random.default_rng(seed)
    cells = [8 * r + c for r in range(7) for c in range(7)]
    occ_me = np.zeros(n, np.uint64)
    occ_op = np.zeros(n, np.uint64)
    cells_me = np.zeros(n, np.uint64)
    for i in range(n):
        pick = rng.permutation(cells)
        mine, empty = pick[:6], pick[6:6 + int(rng.integers(0, 9))]
        occ_me[i] = sum(1 << int(c) for c in mine)
        occ_op[i] = sum(1 << int(c) for c in cells if c not in mine and c not in empty)
        cells_me[i] = sum(int(c) << (8 * k) for k, c in enumerate(mine))
    return occ_me, occ_op, cells_me, rng.integers(0, 2 ** 32, size=n, dtype=np.uint32)


@pytest.mark.parametrize("wide", [1, 0], ids=["wide", "tri"])
def test_spec_pick_boxed_in(sp, wide):
    """the exact path's outcomes: a pass (no checker can move), some checkers that cannot move, a checker without a walk"""
    arrays = [np.ascontiguousarray(a) for a in boxed_boards(20000, seed=47)]
    out = np.zeros(5, dtype=np.int64)
    sp.sp_check_boards(*(a.ctypes.data_as(ctypes.c_void_p) for a in arrays), arrays[0].size, wide,
                       out.ctypes.data_as(ctypes.c_void_p))
    bad, starts, fallback, passes, stuck = report(out)
    assert bad == 0
    assert passes > 0
    assert stuck > passes                      # some positions have checkers that cannot move next to ones that can
    assert fallback > stuck                    # and some a checker without a walk that can still jump


def test_no_pass_with_six_opponents(sp):
    """exhaustively: no placement of the mover's six checkers is boxed in (no walk, no jump) by six opponents; nine box in
    the two corner triangles, which shows the search finds a box where one exists"""
    assert sp.sp_boxed_in_count(6) == 0
    assert sp.sp_boxed_in_count(9) == 2
