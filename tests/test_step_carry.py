"""The carry-over env step (CCX_STEP_VARIANT=11, kernel k_step_random_carry): k_step_random_pick with each round's flood fill
bounded to K steps and unfinished fills carried into the next round, so that the lanes of a warp may be on different plies.
Each game must still play exactly the moves it plays under the pick-first kernel (variant 10) and the work-queue kernel
(variant 9), and trace its rows at its own ply."""
import numpy as np
import pytest

import oracle as orc
from test_step_pick_first import near_win_states

SEED = 0x5EED2026


@pytest.fixture(scope="module")
def eng():
    from chinesecheckersagent_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def gpu_run(eng, monkeypatch, variant, n, plies, chunks=1, state=None, trace_games=0):
    import torch
    from chinesecheckersagent_b200.engine import BatchedEnv
    monkeypatch.setenv("CCX_STEP_VARIANT", str(variant))
    env = BatchedEnv(n, engine=eng, seed=SEED, game_id0=11, state=state)
    traces = [env.step_random(plies // chunks, trace_games=trace_games) for _ in range(chunks)]
    torch.cuda.synchronize()
    return env.state[:5].clone(), env.wins.clone(), traces


# one wave is 148 x 448 = 66,304 games: 66,304 runs the one-block-per-SM instantiation, 66,305 the two-blocks-per-SM one
@pytest.mark.gpu
@pytest.mark.parametrize("n,plies", [(65536, 1024), (300000, 256), (1, 256), (31, 256), (66304, 256), (66305, 256)])
def test_carry_kernel_matches_pick_and_work_queue_kernels(eng, monkeypatch, n, plies):
    import torch
    st, wins, _ = gpu_run(eng, monkeypatch, 11, n, plies)
    for ref in (10, 9):
        ref_st, ref_wins, _ = gpu_run(eng, monkeypatch, ref, n, plies)
        assert torch.equal(st, ref_st), ref
        assert torch.equal(wins, ref_wins), ref


@pytest.mark.gpu
@pytest.mark.parametrize("n", [66304, 66305])
def test_carry_kernel_matches_with_wins(eng, monkeypatch, n):
    import torch
    st0 = near_win_states(n, seed=3)
    st, wins, _ = gpu_run(eng, monkeypatch, 11, n, 256, state=st0)
    for ref in (10, 9):
        ref_st, ref_wins, _ = gpu_run(eng, monkeypatch, ref, n, 256, state=st0)
        assert torch.equal(st, ref_st), ref
        assert torch.equal(wins, ref_wins), ref
    assert int(wins.min()) > 0


@pytest.mark.gpu
def test_carry_kernel_chunking_invariant(eng, monkeypatch):
    import torch
    a = gpu_run(eng, monkeypatch, 11, 65536, 512)
    b = gpu_run(eng, monkeypatch, 11, 65536, 512, chunks=2)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["start", "near_win"])
def test_carry_kernel_trace_matches_oracle(eng, monkeypatch, kind):
    # more games than traced ones, so that warps mix traced and untraced lanes
    n, tg = 5000, 1536
    if kind == "start":
        st0, plies = orc.start_states(n), 200
    else:
        st0, plies = near_win_states(n, seed=7), 60
    st, wins, (trace,) = gpu_run(eng, monkeypatch, 11, n, plies, state=st0, trace_games=tg)
    ost, owins, otrace = orc.step_random(st0, SEED, 0, plies, game_id0=11, trace_games=tg, nthreads=8)
    got = trace.cpu().numpy().view(np.uint64)
    for t in range(plies):
        assert np.array_equal(got[t], otrace[t]), t
    assert np.array_equal(st.cpu().numpy().view(np.uint64), ost[:5])
    assert np.array_equal(wins.cpu().numpy().view(np.uint64), owins)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["0", "8", "12", "x"])
def test_unknown_step_variants_are_errors(eng, monkeypatch, variant):
    from chinesecheckersagent_b200 import _lib
    from chinesecheckersagent_b200.engine import BatchedEnv
    env = BatchedEnv(64, engine=eng, seed=SEED)
    monkeypatch.setenv("CCX_STEP_VARIANT", variant)
    with pytest.raises(_lib.CcxError):
        env.step_random(4)
