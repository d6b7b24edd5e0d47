"""The ply of the carry-over env step (k_step_random_carry): its selects (select64_step, the rank table sel7_rank) against
select64, and a host build of its whole ply (carry_ply_start / fill_step / carry_ply_to, with the occupancy carried through
the fill as the kernel carries it) against the oracle.  CPU only: nvcc builds the kernel's source for the host."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle as orc
from test_step_pick_first import near_win_states, rare_checkers

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "carry_ply.cu")
SEED = 0x5EED2026
VALID = 0x007F7F7F7F7F7F7F


@pytest.fixture(scope="module")
def cp(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("carry_ply") / "libcarry_ply.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-cudart", "none", "-o", lib, SRC], env=env)
    L = ctypes.CDLL(lib)
    vp, i64, i32, u64, u32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64, ctypes.c_uint32
    L.cp_select64.argtypes = [vp, vp, i64, vp, vp]
    L.cp_select64.restype = None
    L.cp_sel7.argtypes = [vp]
    L.cp_sel7.restype = None
    L.cp_step_random.argtypes = [vp, i64, i64, u64, u32, i32, vp, vp, i64]
    L.cp_step_random.restype = None
    return L


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def select_both(cp, m, k):
    m = np.ascontiguousarray(m, dtype=np.uint64)
    k = np.ascontiguousarray(k, dtype=np.uint32)
    fast = np.empty(m.size, np.int32)
    ref = np.empty(m.size, np.int32)
    cp.cp_select64(P(m), P(k), m.size, P(fast), P(ref))
    return fast, ref


def every_rank(masks):
    """each mask repeated once per set bit, with ranks 0 .. popc - 1"""
    masks = np.asarray(masks, dtype=np.uint64)
    cnt = np.bitwise_count(masks).astype(np.int64)
    m = np.repeat(masks, cnt)
    k = np.arange(m.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    return m, k.astype(np.uint32)


def test_rank_table_every_value_and_rank(cp):
    """the checker select: every 6-bit movable mask (and every 7-bit byte of a destination mask) at every rank"""
    out = np.empty(128 * 7, np.int32)
    cp.cp_sel7(P(out))
    out = out.reshape(128, 7)
    for v in range(128):
        bits = [b for b in range(7) if (v >> b) & 1]
        assert list(out[v, :len(bits)]) == bits, v
    m, k = every_rank(np.arange(1, 64))
    fast, ref = select_both(cp, m, k)
    assert np.array_equal(out[m.astype(np.int64), k.astype(np.int64)], ref)


def test_select64_step_random_masks(cp):
    rng = np.random.default_rng(SEED)
    full = rng.integers(0, 2 ** 64, size=1 << 20, dtype=np.uint64, endpoint=False)
    sparse = full & rng.integers(0, 2 ** 64, size=full.size, dtype=np.uint64) & rng.integers(0, 2 ** 64, size=full.size, dtype=np.uint64)
    board = full & np.uint64(VALID)                      # destination masks: on-board cells only
    for masks in (full, sparse, board):
        masks = masks[masks != 0]
        cnt = np.bitwise_count(masks).astype(np.uint64)
        k = (rng.integers(0, 2 ** 32, size=masks.size, dtype=np.uint64) * cnt >> np.uint64(32)).astype(np.uint32)
        fast, ref = select_both(cp, masks, k)
        assert np.array_equal(fast, ref)


def test_select64_step_extreme_masks(cp):
    """masks with 1, 2, 63 and 64 bits set, and whole / nearly whole boards, at every rank"""
    one = [1 << a for a in range(64)]
    two = [(1 << a) | (1 << b) for a in range(64) for b in range(a + 1, 64)]
    all64 = (1 << 64) - 1
    many = [all64] + [all64 ^ (1 << a) for a in range(64)]
    board = [VALID] + [VALID ^ (1 << a) for a in range(64) if (VALID >> a) & 1]
    m, k = every_rank(np.array(one + two + many + board, dtype=np.uint64))
    fast, ref = select_both(cp, m, k)
    assert np.array_equal(fast, ref)


def host_step(cp, st, seed, step0, plies, game_id0):
    st = np.array(st, dtype=np.uint64, order="C")
    n = st.shape[1]
    wins = np.zeros(2, dtype=np.uint64)
    trace = np.zeros((plies, n, orc.TRACE_WORDS), dtype=np.uint64)
    cp.cp_step_random(P(st), n, game_id0, seed, step0, plies, P(wins), P(trace), n)
    return st, wins, trace


@pytest.mark.parametrize("kind", ["start", "crowded", "near_win"])
def test_carry_ply_host_matches_oracle(cp, kind):
    if kind == "start":                       # steady-state random play from the start position, won games restart
        st, plies, step0, gid0 = orc.start_states(2000), 300, 17, 123
    elif kind == "crowded":                   # Board(randomised=True) placements: checkers boxed in far from the corners
        st, plies, step0, gid0 = orc.random_states(3000, seed=29), 50, 0, 5000
    else:
        st, plies, step0, gid0 = near_win_states(2000, seed=31), 60, 9, 77
    got, gwins, gtrace = host_step(cp, st, SEED, step0, plies, gid0)
    ost, owins, otrace = orc.step_random(st, SEED, step0, plies, game_id0=gid0, trace_games=st.shape[1], nthreads=8)
    assert np.array_equal(got[:5], ost[:5])
    assert np.array_equal(gwins, owins)
    assert np.array_equal(gtrace, otrace)
    jump_only, stuck = rare_checkers(otrace)
    assert jump_only > 0 and stuck > 0, (jump_only, stuck)
    if kind == "near_win":
        assert owins.min() > 0, owins
