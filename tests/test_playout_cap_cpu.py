"""CPU checks of the playout cap draw's host restatement (tests/playout_cap_ref.py): its full share follows p, and its Philox
counter word never meets the resignation probe's."""
import math

import numpy as np
import pytest

import playout_cap_ref as pc


@pytest.mark.parametrize("p", [0.0, 0.25, 0.5, 1.0])
def test_full_share_is_binomial(p):
    slots = np.arange(0, 400, dtype=np.uint64) * np.uint64(0x10001) + np.uint64(7 << 32)
    full = 0
    draws = 0
    for serial, ply in [(0, 6), (1, 7), (3, 40), (9, 101)]:
        f = pc.full_search(0x1234ABCD5678EF01, slots, serial, ply, p)
        full += int(f.sum())
        draws += f.size
    sd = math.sqrt(draws * p * (1 - p))
    assert abs(full - draws * p) <= 4 * sd, (full, draws)


def test_draw_is_a_function_of_game_and_ply():
    a = pc.full_search(5, [3, 4, 5], 2, 10, 0.5)
    b = pc.full_search(5, [3, 4, 5], 2, 10, 0.5)
    assert np.array_equal(a, b)
    x = [pc.full_search(5, list(range(64)), s, ply, 0.5) for s, ply in [(2, 10), (3, 10), (2, 11)]]
    assert not np.array_equal(x[0], x[1]) and not np.array_equal(x[0], x[2])


def test_counter_word_never_meets_the_resignation_probe():
    words = {pc.counter_word(ply) for ply in range(1 << 16)}
    assert pc.RESIGN_PURPOSE not in words
