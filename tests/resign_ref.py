"""Host restatement of the self-play resignation rule of include/ccx.h (ccx_selfplay_resign): the resign value r of one root in
the kernel's float64 summation order, the per-player streak and the windowed minimum the calibration samples hold."""
import math


def resign_value(N, Q):
    """r = max(sum N*Q / sum N, Q of the first edge with the maximal N) over a root's edges in edge order; lane l of a warp sums
    edges l + 32c (c = 0..3, 0.0 past the last edge), then an xor butterfly over 16, 8, 4, 2, 1.  NaN when sum N = 0."""
    ne = len(N)
    assert ne <= 128
    nq, nn = [0.0] * 32, [0.0] * 32
    for lane in range(32):
        for c in range(4):
            j = lane + 32 * c
            n = float(N[j]) if j < ne else 0.0
            q = float(Q[j]) if j < ne else 0.0
            nq[lane] = nq[lane] + n * q
            nn[lane] = nn[lane] + n
    for off in (16, 8, 4, 2, 1):
        nq = [nq[lane] + nq[lane ^ off] for lane in range(32)]
        nn = [nn[lane] + nn[lane ^ off] for lane in range(32)]
    if nn[0] == 0.0:
        return math.nan
    best = 0
    for j in range(ne):
        if N[j] > N[best]:
            best = j
    return max(nq[0] / nn[0], float(Q[best]))


class PlayerTrack:
    """one player's streak and window over its searched plies"""

    def __init__(self, plies):
        self.plies, self.streak, self.last, self.wmin = plies, 0, [], math.inf

    def push(self, r, threshold):
        """add one searched ply's r; True when the streak reaches `plies` at this ply"""
        self.last = (self.last + [r])[-self.plies:]
        if len(self.last) == self.plies:
            self.wmin = min(self.wmin, max(self.last))
        self.streak = min(self.streak + 1, self.plies) if r < threshold else 0
        return self.streak >= self.plies


def track_game(values, threshold, plies, probe):
    """values: [(player 0/1, r)] of one game's searched plies in order.  Returns (index of the ply at which the game resigns or
    None, player who would have resigned first or None, [window minimum of player 0, of player 1]).  A probe never resigns:
    every ply is tracked; otherwise tracking stops at the resignation."""
    tr = [PlayerTrack(plies), PlayerTrack(plies)]
    resign_at, would = None, None
    for k, (p, r) in enumerate(values):
        if tr[p].push(r, threshold):
            if would is None:
                would = p
            if not probe:
                resign_at = k
                break
    return resign_at, would, [tr[0].wmin, tr[1].wmin]
