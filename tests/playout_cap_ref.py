"""Host restatement of the self-play playout cap draw of include/ccx.h (ccx_selfplay_playout_cap): a searched ply is a full
search when x / 2^32 < p, x = the first word of Philox4x32-10 with key (seed lo, seed hi) and counter (slot id lo, slot id hi,
serial lo, 0x50430000 + ply)."""
import numpy as np

from symmetry_ref import philox_x

PURPOSE = 0x50430000
RESIGN_PURPOSE = 0x52534750


def counter_word(ply):
    return PURPOSE + int(ply)


def full_search(seed, slot_id, serial, ply, p):
    """True when the searched ply `ply` of game (slot_id, serial) gets the full search; vectorised over slot_id"""
    sid = np.asarray(slot_id, dtype=np.uint64)
    lo, hi = sid & np.uint64(0xFFFFFFFF), sid >> np.uint64(32)
    x = np.array([int(philox_x(seed & 0xFFFFFFFF, seed >> 32, int(a), int(b), int(serial) & 0xFFFFFFFF, counter_word(ply)))
                  for a, b in zip(np.atleast_1d(lo), np.atleast_1d(hi))], dtype=np.float64)
    return x / 4294967296.0 < p
