"""NumPy restatement of the mirror-symmetric net evaluation (include/ccx.h ccx_net_set_symmetry): the mirror of states,
planes and policy indices, the random orientation's key and hash, and how a mode turns raw net rows into (p, v).  The CPU
tests check it against the oracle; the GPU tests compare the engine against it bit for bit."""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
SYM_COUNTER = 0x53594D
MODES = {"off": 0, "random": 1, "mean": 2}


def mirror_cell8(b):
    """bit index 8 r + c -> 8 (6 - c) + (6 - r); 0xFF (no cell) stays"""
    b = int(b)
    if b == 0xFF:
        return b
    r, c = b >> 3, b & 7
    return 8 * (6 - c) + (6 - r)


MIRROR_ACTION = np.array([k * 49 + (6 - (a % 7)) * 7 + (6 - a // 7) for k in range(6) for a in range(49)], dtype=np.int64)


def mirror_planes(bx):
    """(N, 7, 7, 7) planes of each position mirrored: out[r', c'] = in[6 - c', 6 - r'] (utils.augment_train_data's map)"""
    return np.ascontiguousarray(np.asarray(bx)[:, ::-1, ::-1, :].transpose(0, 2, 1, 3))


def _mirror_bytes(w, nbytes):
    out = 0
    for k in range(nbytes):
        out |= mirror_cell8((w >> (8 * k)) & 0xFF) << (8 * k)
    return out


def mirror_state(st):
    """uint64 [8][n] states mirrored: occupancies, checker cells (ids kept), the last two moves and the destination history;
    ply count, side to move, status and the self-play word unchanged"""
    st = np.asarray(st, dtype=np.uint64)
    out = st.copy()
    for i in range(st.shape[1]):
        for w in (0, 1):
            occ, m = int(st[w, i]), 0
            while occ:
                b = occ & -occ
                m |= 1 << mirror_cell8(b.bit_length() - 1)
                occ ^= b
            out[w, i] = m
        for w in (2, 3, 5, 6):
            out[w, i] = _mirror_bytes(int(st[w, i]), 8 if w >= 5 else 6) | (int(st[w, i]) & (0xFFFF << 48 if w < 5 else 0))
        meta = int(st[4, i])
        out[4, i] = (meta & ~0xFFFFFFFF) | _mirror_bytes(meta & 0xFFFFFFFF, 4)
    return out


def philox_x(k0, k1, c0, c1, c2=0, c3=0):
    """Philox4x32-10, first output word, vectorised over c0 (numpy uint64 holding 32-bit values)"""
    c0 = np.asarray(c0, dtype=np.uint64) & M32
    c1 = np.full_like(c0, c1)
    c2 = np.full_like(c0, c2)
    c3 = np.full_like(c0, c3)
    k0, k1 = np.uint64(k0 & 0xFFFFFFFF), np.uint64(k1 & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & M32, p0 & M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c0


def position_hash(st):
    """h(s) = fold32(OCC1 * 0x9E3779B97F4A7C15 + OCC2 * 0xC2B2AE3D27D4EB4F + (META & 0xFFFFFFFFFFFF)) per column of [>=5][n]"""
    st = np.asarray(st, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = st[0] * np.uint64(0x9E3779B97F4A7C15) + st[1] * np.uint64(0xC2B2AE3D27D4EB4F) + (st[4] & np.uint64(0xFFFFFFFFFFFF))
    return (z >> np.uint64(32)) ^ (z & M32)


def mirrored(st, seed):
    """the random mode's orientation of each position: True = evaluated mirrored"""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return (philox_x(seed & 0xFFFFFFFF, seed >> 32, position_hash(st), SYM_COUNTER) & np.uint64(1)).astype(bool)


def net_rows(planes, mode, flags=None):
    """the net batch a mode evaluates for planes (n, 7, 7, 7): random = row i mirrored where flags[i]; mean = rows 2i (as is)
    and 2i + 1 (mirrored)"""
    planes = np.asarray(planes)
    if mode == MODES["random"]:
        out = planes.copy()
        out[flags] = mirror_planes(planes[flags])
        return out
    if mode == MODES["mean"]:
        out = np.empty((2 * len(planes),) + planes.shape[1:], planes.dtype)
        out[0::2], out[1::2] = planes, mirror_planes(planes)
        return out
    return planes


def combine(p_rows, v_rows, mode, flags=None):
    """(p float64 [n][294], v float64 [n]) from the softmax p_rows and float64 values v_rows of net_rows' batch"""
    p_rows, v_rows = np.asarray(p_rows, np.float64), np.asarray(v_rows, np.float64)
    if mode == MODES["random"]:
        p = p_rows.copy()
        p[np.ix_(flags, MIRROR_ACTION)] = p_rows[flags]           # p[mirror(i)] = softmax(mirrored logits)[i]
        return p, v_rows.copy()
    if mode == MODES["mean"]:
        p = (p_rows[0::2] + p_rows[1::2][:, MIRROR_ACTION]) * 0.5
        v = (v_rows[0::2] + v_rows[1::2]) * 0.5
        return p, v
    return p_rows, v_rows
