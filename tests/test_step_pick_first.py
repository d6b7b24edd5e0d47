"""The pick-first env step (pick_random_first in ccx_device.cuh, kernel k_step_random_pick): the random-legal ply that
decides the checker before it flood-fills any jumps, and then fills the picked checker's jumps only.  The CPU tests step
a host build of the same source and compare it with the oracle; the GPU tests compare the kernel with the work-queue
kernel that computes all six destination sets (CCX_STEP_VARIANT=9)."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle as orc

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "pick_first.cu")
SEED = 0x5EED2026


@pytest.fixture(scope="module")
def pf(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("pick_first") / "libpick_first.so")
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call([nvcc, "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                           "-shared", "-cudart", "none", "-o", lib, SRC], env=env)
    L = ctypes.CDLL(lib)
    vp, i64, i32, u64, u32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_uint64, ctypes.c_uint32
    L.pf_step_random.argtypes = [vp, i64, i64, u64, u32, i32, vp, vp, i64]
    L.pf_step_random.restype = None
    return L


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def host_step(pf, st, seed, step0, plies, game_id0):
    st = np.array(st, dtype=np.uint64, order="C")
    n = st.shape[1]
    wins = np.zeros(2, dtype=np.uint64)
    trace = np.zeros((plies, n, orc.TRACE_WORDS), dtype=np.uint64)
    pf.pf_step_random(P(st), n, game_id0, seed, step0, plies, P(wins), P(trace), n)
    return st, wins, trace


def neighbour_table():
    nb = np.zeros(64, dtype=np.uint64)
    for r in range(7):
        for c in range(7):
            m = 0
            for dr, dc in ((-1, 0), (0, 1), (1, 1), (1, 0), (0, -1), (-1, -1)):     # board.py:33-40
                if 0 <= r + dr < 7 and 0 <= c + dc < 7:
                    m |= 1 << (8 * (r + dr) + c + dc)
            nb[8 * r + c] = m
    return nb


def near_win_states(n, seed):
    """Random play from the start almost never wins, so these positions put five checkers of one side on its target
    triangle and the sixth anywhere: games are won within a few plies and restart, which exercises the win / reset path."""
    rng = np.random.default_rng(seed)
    targets = ([(0, 4), (0, 5), (0, 6), (1, 5), (1, 6), (2, 6)], [(4, 0), (5, 0), (6, 0), (5, 1), (6, 1), (6, 2)])   # board.py:96-111
    st = np.zeros((orc.STATE_WORDS, n), dtype=np.uint64)
    cells = [(r, c) for r in range(7) for c in range(7)]
    for i in range(n):
        p = int(rng.integers(0, 2))
        mine = [targets[p][k] for k in rng.permutation(6)[:5]]
        free = [x for x in cells if x not in targets[p]]
        pick = rng.choice(len(free), size=7, replace=False)
        mine.append(free[pick[0]])
        other = [free[k] for k in pick[1:]]
        order = rng.permutation(6)
        mine = [mine[k] for k in order]
        st[:, i] = orc.pack_state(*((mine, other) if p == 0 else (other, mine)), to_move=int(rng.integers(0, 2)))
    return st


def rare_checkers(trace):
    """From oracle trace rows: (checkers with no empty neighbour that can still jump, checkers that cannot move at all)."""
    rows = trace.reshape(-1, orc.TRACE_WORDS)
    p2 = ((rows[:, 4] >> np.uint64(48)) & np.uint64(1)).astype(bool)
    cells = np.where(p2, rows[:, 3], rows[:, 2])
    occ = rows[:, 0] | rows[:, 1]
    nb = neighbour_table()
    jump_only = stuck = 0
    for k in range(6):
        cell = ((cells >> np.uint64(8 * k)) & np.uint64(0x3F)).astype(np.int64)
        walk = nb[cell] & ~occ
        dest = rows[:, 5 + k]
        jump_only += int(((walk == 0) & (dest != 0)).sum())
        stuck += int((dest == 0).sum())
    return jump_only, stuck


@pytest.mark.parametrize("kind", ["start", "crowded", "near_win"])
def test_pick_first_host_matches_oracle(pf, kind):
    if kind == "start":                       # steady-state random play from the start position, won games restart
        st, plies, step0, gid0 = orc.start_states(2000), 300, 17, 123
    elif kind == "crowded":                   # Board(randomised=True) placements: checkers boxed in far from the corners
        st, plies, step0, gid0 = orc.random_states(3000, seed=29), 50, 0, 5000
    else:
        st, plies, step0, gid0 = near_win_states(2000, seed=31), 60, 9, 77
    got, gwins, gtrace = host_step(pf, st, SEED, step0, plies, gid0)
    ost, owins, otrace = orc.step_random(st, SEED, step0, plies, game_id0=gid0, trace_games=st.shape[1], nthreads=8)
    assert np.array_equal(got[:5], ost[:5])
    assert np.array_equal(gwins, owins)
    # from / to / checker id / winner of every ply, and the six destination sets the trace rows carry
    assert np.array_equal(gtrace, otrace)
    jump_only, stuck = rare_checkers(otrace)
    assert jump_only > 0 and stuck > 0, (jump_only, stuck)
    if kind == "near_win":
        assert owins.min() > 0, owins


# ---- GPU: the kernel against the all-six-closures work-queue kernel --------------------------------------------------

@pytest.fixture(scope="module")
def eng():
    from chinesecheckersagent_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def gpu_run(eng, n, plies, chunks=1, state=None):
    import torch
    from chinesecheckersagent_b200.engine import BatchedEnv
    env = BatchedEnv(n, engine=eng, seed=SEED, game_id0=11, state=state)
    for _ in range(chunks):
        env.step_random(plies // chunks)
    torch.cuda.synchronize()
    return env.state[:5].clone(), env.wins.clone()


@pytest.mark.gpu
@pytest.mark.parametrize("n,plies", [(65536, 1024), (300000, 256), (1, 256), (31, 256), (66305, 256)])
def test_pick_first_kernel_matches_work_queue_kernel(eng, monkeypatch, n, plies):
    import torch
    monkeypatch.delenv("CCX_STEP_VARIANT", raising=False)
    st, wins = gpu_run(eng, n, plies)
    monkeypatch.setenv("CCX_STEP_VARIANT", "9")
    ref_st, ref_wins = gpu_run(eng, n, plies)
    assert torch.equal(st, ref_st)
    assert torch.equal(wins, ref_wins)


@pytest.mark.gpu
def test_pick_first_kernel_matches_work_queue_kernel_with_wins(eng, monkeypatch):
    import torch
    st0 = near_win_states(66305, seed=3)
    monkeypatch.delenv("CCX_STEP_VARIANT", raising=False)
    st, wins = gpu_run(eng, st0.shape[1], 256, state=st0)
    monkeypatch.setenv("CCX_STEP_VARIANT", "9")
    ref_st, ref_wins = gpu_run(eng, st0.shape[1], 256, state=st0)
    assert torch.equal(st, ref_st)
    assert torch.equal(wins, ref_wins)
    assert int(wins.min()) > 0


@pytest.mark.gpu
def test_pick_first_kernel_chunking_invariant(eng, monkeypatch):
    import torch
    monkeypatch.delenv("CCX_STEP_VARIANT", raising=False)
    a = gpu_run(eng, 65536, 256)
    b = gpu_run(eng, 65536, 256, chunks=4)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_unknown_step_variant_is_an_error(eng, monkeypatch):
    from chinesecheckersagent_b200 import _lib
    monkeypatch.setenv("CCX_STEP_VARIANT", "5")
    with pytest.raises(_lib.CcxError):
        gpu_run(eng, 64, 4)
