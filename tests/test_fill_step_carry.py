"""The carry-over env step's fill (k_step_random_carry): the per-cell constants it computes with ALU instructions
(carry_cell) against the table the other kernels load (tri_cell_info), and its fill (carry_fill_start, which takes the
first step, then fill_step_carry) against fill_start / fill_step, closure by closure.  CPU only: nvcc builds the kernel's
source for the host."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle as orc
from test_step_pick_first import near_win_states

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "fill_carry.cu")
SEED = 0x5EED2026
VALID = 0x007F7F7F7F7F7F7F
NLP = 29                                   # answer columns per occupancy pattern of the diagonal table (CCX_JT3_NLP)


@pytest.fixture(scope="module")
def fc(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("fill_carry") / "libfill_carry.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-cudart", "none", "-o", lib, SRC], env=env)
    L = ctypes.CDLL(lib)
    vp, i64 = ctypes.c_void_p, ctypes.c_int64
    L.fc_cell_info.argtypes = [vp]
    L.fc_cell_info.restype = None
    L.fc_prmt.argtypes = [vp, vp, vp, i64, vp]
    L.fc_prmt.restype = None
    L.fc_diag_answer.argtypes = [ctypes.c_int, ctypes.c_uint64]
    L.fc_diag_answer.restype = ctypes.c_uint64
    L.fc_closures.argtypes = [vp, vp, i64, vp]
    L.fc_closures.restype = i64
    return L


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def prmt(fc, lo, hi, sel):
    lo, hi, sel = (np.ascontiguousarray(a, dtype=np.uint32) for a in (lo, hi, sel))
    out = np.empty(lo.size, np.uint32)
    fc.fc_prmt(P(lo), P(hi), P(sel), lo.size, P(out))
    return out


def test_prmt_host_model(fc):
    """the host model of PRMT: bytes by nibble, a nibble with bit 3 set replicates the byte's sign"""
    rng = np.random.default_rng(SEED)
    lo, hi, sel = (rng.integers(0, 2 ** 32, size=4096, dtype=np.uint64).astype(np.uint32) for _ in range(3))
    got = prmt(fc, lo, hi, sel)
    v = lo.astype(np.uint64) | (hi.astype(np.uint64) << np.uint64(32))
    want = np.zeros(lo.size, np.uint64)
    for q in range(4):
        n = (sel.astype(np.uint64) >> np.uint64(4 * q)) & np.uint64(15)
        b = (v >> (np.uint64(8) * (n & np.uint64(7)))) & np.uint64(0xFF)
        b = np.where(n & np.uint64(8), np.where(b & np.uint64(0x80), np.uint64(0xFF), np.uint64(0)), b)
        want |= b << np.uint64(8 * q)
    assert np.array_equal(got, want.astype(np.uint32))


def test_cell_constants_equal_tri_cell_info(fc):
    """every on-board cell: the row / column selectors, the diagonal's byte, shift and answer column equal tri_cell_info's;
    on the four corner diagonals (no jump possible) the diagonal selector picks a zero byte and the column is in range"""
    out = np.zeros(64 * 7, np.uint64)
    fc.fc_cell_info(P(out))
    out = out.reshape(64, 7).astype(np.int64)
    rng = np.random.default_rng(SEED)
    words = rng.integers(0, 2 ** 64, size=256, dtype=np.uint64) & np.uint64(VALID)   # guard bits (bit 7 of each byte) clear
    wlo, whi = (words & np.uint64(0xFFFFFFFF)).astype(np.uint32), (words >> np.uint64(32)).astype(np.uint32)
    corners = 0
    for c in range(64):
        if not (VALID >> c) & 1:
            continue
        r, col = c >> 3, c & 7
        lo, hi, rsel, csel, dsel, lp8, sh = out[c]
        assert rsel == hi & 0xFFFF and csel == hi >> 16, c
        assert sh == (lo >> 16) & 0xFF, c
        got = prmt(fc, wlo, whi, np.full(words.size, dsel))
        if abs(col - r) <= 4:
            assert lp8 == lo >> 24, c
            assert np.array_equal(got, prmt(fc, wlo, whi, np.full(words.size, lo & 0xFFFF))), c
        else:
            corners += 1
            assert not got.any(), c
            assert 0 <= lp8 <= 8 * (NLP - 1), c
            assert fc.fc_diag_answer(c, VALID) == 0, c
    assert corners == 6


def closures(fc, occ, mover):
    occ = np.ascontiguousarray(occ, dtype=np.uint64)
    mover = np.ascontiguousarray(mover, dtype=np.uint64)
    pairs = ctypes.c_int64(0)
    bad = fc.fc_closures(P(occ), P(mover), occ.size, ctypes.byref(pairs))
    return bad, pairs.value


def test_fill_random_occupancies(fc):
    """2^20 seeded occupancies (sparse, half and dense boards), each with every on-board cell as the mover"""
    rng = np.random.default_rng(SEED)
    n = 1 << 20
    a, b, c = (rng.integers(0, 2 ** 64, size=n, dtype=np.uint64) for _ in range(3))
    occ = np.concatenate([(a & b & c)[: n // 4], (a & b)[n // 4: n // 2], a[n // 2: 3 * n // 4], (a | b)[3 * n // 4:]])
    bad, pairs = closures(fc, occ, np.full(n, VALID, np.uint64))
    assert pairs > 40 * n
    assert bad == 0


@pytest.mark.parametrize("kind", ["start", "crowded", "near_win"])
def test_fill_game_positions(fc, kind):
    """positions met in random play, Board(randomised=True) placements and near-win positions; every checker of both sides
    as the mover"""
    if kind == "start":
        st, _, _ = orc.step_random(orc.start_states(4000), SEED, 0, 300, nthreads=8)
    elif kind == "crowded":
        st = orc.random_states(20000, seed=29)
    else:
        st = near_win_states(20000, seed=31)
    occ = st[0] | st[1]
    bad, pairs = closures(fc, occ, occ)
    assert pairs == 12 * occ.size
    assert bad == 0
