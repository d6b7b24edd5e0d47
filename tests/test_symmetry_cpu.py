"""CPU checks of the mirror symmetry that ccx_net_set_symmetry relies on, and of the NumPy restatement of its modes
(tests/symmetry_ref.py) that the GPU tests compare the engine against.

The mirror is cell (r, c) -> (6 - c, 6 - r).  On about 10^4 seeded positions of the CPU oracle (random play from the start,
randomised placements advanced by random play, crowded centres, near-win and won positions) it maps legal moves to legal
moves, keeps check_win, and to_model_input of the mirrored position is the planes mirrored, history and side-to-move planes
included."""
import numpy as np

import oracle as orc
import symmetry_ref as sr


def _positions():
    rng = np.random.default_rng(2026)
    parts = []
    start = orc.start_states(2048)
    for k, plies in enumerate((1, 2, 3, 7, 20, 60, 150)):                 # random play from the start (auto-reset on a win)
        parts.append(orc.step_random(start[:, :256], seed=11 + k, step0=0, plies=plies, game_id0=256 * k)[0])
    rnd = orc.random_states(2048, seed=7)
    parts.append(rnd)
    parts.append(orc.step_random(rnd, seed=5, step0=0, plies=9)[0])       # randomised placements advanced by 9 plies
    parts.append(orc.step_random(rnd[:, :1024], seed=6, step0=0, plies=1)[0])
    crowded = np.zeros((orc.STATE_WORDS, 1536), dtype=np.uint64)          # 12 checkers packed into the 4 x 4 centre
    centre = [(r, c) for r in range(1, 5) for c in range(1, 5)]
    for i in range(crowded.shape[1]):
        pick = rng.choice(len(centre), size=12, replace=False)
        pos = [centre[j] for j in pick]
        crowded[:, i] = orc.pack_state(pos[:6], pos[6:], to_move=int(rng.integers(0, 2)), ply=int(rng.integers(0, 40)))
    parts.append(crowded)
    parts.append(orc.step_random(crowded, seed=8, step0=0, plies=2)[0])
    near = np.zeros((orc.STATE_WORDS, 1024), dtype=np.uint64)             # one or no checker away from the target triangle
    cells = [(r, c) for r in range(7) for c in range(7)]
    for i in range(near.shape[1]):
        me, tgt = (orc.START_P1, orc.START_P2) if i % 2 == 0 else (orc.START_P2, orc.START_P1)
        keep = list(tgt) if i % 8 == 0 else [tgt[j] for j in rng.permutation(6)[:5]]
        rest = [c for c in cells if c not in keep]
        extra = [rest[j] for j in rng.choice(len(rest), size=12 - len(keep), replace=False)]
        mine = keep + extra[:6 - len(keep)]
        other = extra[6 - len(keep):]
        p1, p2 = (mine, other) if i % 2 == 0 else (other, mine)
        near[:, i] = orc.pack_state(p1, p2, to_move=int(rng.integers(0, 2)), ply=int(rng.integers(2, 90)),
                                    last_moves=[(rest[0], p1[0]), (rest[1], p2[0])][:int(rng.integers(0, 3))])
    parts.append(near)
    return np.ascontiguousarray(np.concatenate(parts, axis=1))


def _mirror_mask(m):
    out, m = 0, int(m)
    while m:
        b = m & -m
        out |= 1 << sr.mirror_cell8(b.bit_length() - 1)
        m ^= b
    return out


def test_mirror_maps_are_involutions_and_match_augmentation():
    from chinesecheckersagent_b200 import utils
    assert np.array_equal(sr.MIRROR_ACTION[sr.MIRROR_ACTION], np.arange(294))
    assert sorted(sr.MIRROR_ACTION) == list(range(294))
    for b in [8 * r + c for r in range(7) for c in range(7)] + [0xFF]:
        assert sr.mirror_cell8(sr.mirror_cell8(b)) == b
    rng = np.random.default_rng(0)
    bx = rng.integers(0, 7, (16, 7, 7, 7)).astype(np.uint8)
    assert np.array_equal(sr.mirror_planes(sr.mirror_planes(bx)), bx)
    py = rng.random((16, 294))
    ax, ap, _ = utils.augment_train_data(bx, py, np.zeros(16), mirror_pi=True)
    assert np.array_equal(ax[16:], sr.mirror_planes(bx))
    assert np.array_equal(ap[16:], py[:, sr.MIRROR_ACTION])         # augmented pi[b] = pi[mirror(b)]
    st = _positions()[:, ::37]
    assert np.array_equal(sr.mirror_state(sr.mirror_state(st)), st)


def test_oracle_is_mirror_symmetric():
    st = _positions()
    assert st.shape[1] >= 10000
    ms = sr.mirror_state(st)
    start = orc.start_states(1)
    mstart = sr.mirror_state(start)                                     # the start position maps to itself (as a board;
    assert np.array_equal(mstart[[0, 1, 4]], start[[0, 1, 4]])         # the mirror keeps checker ids, so ids 1 and 2 swap cells)
    for w in (2, 3):
        assert sorted(int(mstart[w, 0]) >> (8 * k) & 0xFF for k in range(6)) == sorted(int(start[w, 0]) >> (8 * k) & 0xFF for k in range(6))
    # move generation commutes with the mirror, checker by checker
    masks, mmasks = orc.movegen(st), orc.movegen(ms)
    want = np.vectorize(_mirror_mask, otypes=[object])(masks.astype(object)).astype(np.uint64)
    assert np.array_equal(mmasks, want)
    # check_win is unchanged (and progress counts, which are symmetric too)
    inf, minf = orc.info(st), orc.info(ms)
    assert np.array_equal(inf[:, :3], minf[:, :3])
    assert (inf[:, 0] != 0).sum() >= 100                                 # won positions are among them
    # to_model_input of the mirrored state = the planes mirrored, history and side-to-move planes included
    planes, mplanes = orc.encode(st), orc.encode(ms)
    assert np.array_equal(mplanes, sr.mirror_planes(planes))
    assert planes[..., 2:6].any() and planes[..., 6].any() and not planes[..., 6].all()


def test_restatement_key_hash_and_modes():
    st = _positions()[:, :4096]
    # the hash is the tie rule's root hash, the draw is the oracle's Philox4x32-10 word 0
    for i in (0, 1, 777, 4095):
        z = (int(st[0, i]) * 0x9E3779B97F4A7C15 + int(st[1, i]) * 0xC2B2AE3D27D4EB4F + (int(st[4, i]) & 0xFFFFFFFFFFFF)) % 2 ** 64
        h = (z >> 32) ^ (z & 0xFFFFFFFF)
        assert int(sr.position_hash(st[:, i:i + 1])[0]) == h
        seed = 0x0123456789ABCDEF
        x = orc.philox(seed & 0xFFFFFFFF, seed >> 32, h, sr.SYM_COUNTER, 0, 0)[0]
        assert bool(sr.mirrored(st[:, i:i + 1], seed)[0]) == bool(x & 1)
    f1, f2 = sr.mirrored(st, 1), sr.mirrored(st, 2)
    assert 0.45 < f1.mean() < 0.55 and 0.4 < (f1 != f2).mean() < 0.6
    assert np.array_equal(f1, sr.mirrored(st.copy(), 1))                # a function of (seed, position) only
    # an exactly mirror-equivariant net: both modes give its own output, whatever the orientation
    rng = np.random.default_rng(3)
    n = 64
    p_id = rng.random((n, 294)); p_id /= p_id.sum(1, keepdims=True)
    v_id = rng.random(n) * 2 - 1
    rows = np.empty((2 * n, 294)); rows[0::2] = p_id; rows[1::2] = p_id[:, sr.MIRROR_ACTION]
    vr = np.repeat(v_id, 2)
    p, v = sr.combine(rows, vr, sr.MODES["mean"])
    assert np.array_equal(p, p_id) and np.array_equal(v, v_id)
    flags = rng.random(n) < 0.5
    raw = np.where(flags[:, None], p_id[:, sr.MIRROR_ACTION], p_id)
    p, v = sr.combine(raw, v_id, sr.MODES["random"], flags)
    assert np.array_equal(p, p_id) and np.array_equal(v, v_id)
    # the mean of a net that is not equivariant: element by element, round-to-nearest, then the exact halving
    rows = rng.random((2 * n, 294))
    p, _ = sr.combine(rows, np.zeros(2 * n), sr.MODES["mean"])
    i, a = 5, 123
    assert p[i, a] == (rows[2 * i, a] + rows[2 * i + 1, sr.MIRROR_ACTION[a]]) * 0.5
    planes = rng.integers(0, 7, (n, 7, 7, 7)).astype(np.uint8)
    nr = sr.net_rows(planes, sr.MODES["mean"])
    assert np.array_equal(nr[0::2], planes) and np.array_equal(nr[1::2], sr.mirror_planes(planes))
    nr = sr.net_rows(planes, sr.MODES["random"], flags)
    assert np.array_equal(nr[~flags], planes[~flags]) and np.array_equal(nr[flags], sr.mirror_planes(planes[flags]))
