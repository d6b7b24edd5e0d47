"""The one-wave carry kernel's wide answer tables (build_jump_table_wide: build_jump_table3's row, column and diagonal
answers per cell, already placed on the board) against build_jump_table3's tables plus their shifts, and the expansion, fill
and move generation over them against expand_cell_tri / fill_step / movegen_tri.  CPU only: nvcc builds the kernel's source
for the host."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle as orc
from test_step_pick_first import near_win_states

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "fill_wide.cu")
SEED = 0x5EED2027
VALID = 0x007F7F7F7F7F7F7F
NLP = 29                                   # answer columns per occupancy pattern of the diagonal table (CCX_JT3_NLP)


@pytest.fixture(scope="module")
def fw(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("fill_wide") / "libfill_wide.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-cudart", "none", "-o", lib, SRC], env=env)
    L = ctypes.CDLL(lib)
    vp, i64 = ctypes.c_void_p, ctypes.c_int64
    L.fw_jt3_bytes.restype = i64
    L.fw_wide_words.restype = i64
    L.fw_tables.argtypes = [vp, vp]
    L.fw_tables.restype = None
    L.fw_closures.argtypes = [vp, vp, i64, vp, vp]
    L.fw_closures.restype = i64
    L.fw_movegen.argtypes = [vp, vp, vp, i64]
    L.fw_movegen.restype = i64
    return L


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def diag_column_and_shift(c):
    """build_jump_table3's diagonal answer column of cell c and the diagonal's board shift; None on the corner diagonals"""
    r, col = c >> 3, c & 7
    k = col - r
    if abs(k) > 4:
        return None
    length, pos = 7 - abs(k), (r if k >= 0 else col)
    first = {3: 3 if k > 0 else 0, 4: 6, 5: 10, 6: 15, 7: 21}[length]
    return first + pos, (k if k >= 0 else -8 * k)


def test_wide_entries_equal_shifted_answers(fw):
    """every cell and occupancy pattern: the wide row / column / diagonal entries are build_jump_table3's answers shifted to
    the cell's row, column and diagonal; off-board and corner-diagonal cells hold 0"""
    t3 = np.zeros(fw.fw_jt3_bytes(), np.uint8)
    w = np.zeros(fw.fw_wide_words(), np.uint64)
    fw.fw_tables(P(t3), P(w))
    w = w.reshape(3, 128, 64)
    rows = t3[:128 * 64].reshape(128, 64).astype(np.uint64)
    cols = t3[128 * 64: 2 * 128 * 64].view(np.uint64).reshape(128, 8)
    dias = t3[2 * 128 * 64:].view(np.uint64).reshape(128, NLP)
    assert dias.shape[0] == 128
    corners = 0
    for c in range(64):
        r, col = c >> 3, c & 7
        if not (VALID >> c) & 1:
            assert not w[:, :, c].any(), c
            continue
        assert np.array_equal(w[0, :, c], rows[:, c] << np.uint64(8 * r)), c
        assert np.array_equal(w[1, :, c], cols[:, r] << np.uint64(col)), c
        d = diag_column_and_shift(c)
        if d is None:
            corners += 1
            assert not w[2, :, c].any(), c
        else:
            assert np.array_equal(w[2, :, c], dias[:, d[0]] << np.uint64(d[1])), c
    assert corners == 6
    assert w[0].any() and w[1].any() and w[2].any()


def closures(fw, occ, mover):
    occ = np.ascontiguousarray(occ, dtype=np.uint64)
    mover = np.ascontiguousarray(mover, dtype=np.uint64)
    pairs, steps = ctypes.c_int64(0), ctypes.c_int64(0)
    bad = fw.fw_closures(P(occ), P(mover), occ.size, ctypes.byref(pairs), ctypes.byref(steps))
    return bad, pairs.value, steps.value


def test_wide_fill_random_occupancies(fw):
    """2^20 seeded occupancies (sparse, half and dense boards), each with every on-board cell as the mover"""
    rng = np.random.default_rng(SEED)
    n = 1 << 20
    a, b, c = (rng.integers(0, 2 ** 64, size=n, dtype=np.uint64) for _ in range(3))
    occ = np.concatenate([(a & b & c)[: n // 4], (a & b)[n // 4: n // 2], a[n // 2: 3 * n // 4], (a | b)[3 * n // 4:]])
    bad, pairs, steps = closures(fw, occ, np.full(n, VALID, np.uint64))
    assert pairs > 40 * n and steps > pairs
    assert bad == 0


def game_positions(kind):
    if kind == "start":
        st, _, _ = orc.step_random(orc.start_states(4000), SEED, 0, 300, nthreads=8)
    elif kind == "crowded":
        st = orc.random_states(20000, seed=37)
    else:
        st = near_win_states(20000, seed=41)
    return st


@pytest.mark.parametrize("kind", ["start", "crowded", "near_win"])
def test_wide_fill_game_positions(fw, kind):
    """positions met in random play, Board(randomised=True) placements and near-win positions: every checker of both sides
    as the mover, and the six destination sets of each side (the carry kernel's trace rows)"""
    st = game_positions(kind)
    occ = st[0] | st[1]
    bad, pairs, _ = closures(fw, occ, occ)
    assert pairs == 12 * occ.size
    assert bad == 0
    for me, op, cells in ((st[0], st[1], st[2]), (st[1], st[0], st[3])):
        me, op, cells = (np.ascontiguousarray(x, dtype=np.uint64) for x in (me, op, cells))
        assert fw.fw_movegen(P(me), P(op), P(cells), me.size) == 0
