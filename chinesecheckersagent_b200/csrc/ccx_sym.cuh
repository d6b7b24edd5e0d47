// ccx_sym.cuh — the encode and the float64 softmax of the net evaluation, plain or mirror-symmetric (ccx_net_set_symmetry),
// shared by ccx_net_eval and the fused MCTS round kernels so that both compute the same bits by construction.
//
// The game is symmetric under the anti-diagonal mirror, cell (r, c) -> (6 - c, 6 - r): the start position maps to itself,
// move generation and check_win commute with it, and to_model_input of the mirrored position is the planes mirrored the same
// way (plane 6, the side to move, is constant over the board).  A mirrored evaluation is therefore the net on mirrored planes
// with the policy mapped back, id*49 + r*7 + c -> id*49 + (6-c)*7 + (6-r); no mirrored game state is ever built.
//   SYM_RANDOM: one orientation per position, mirrored when bit 0 of Philox4x32-10 (key = seed, counter = (h(s), 0x53594D, 0, 0))
//               is 1, h(s) = the tie rule's root hash of the position; one net row per position.
//   SYM_MEAN:   both orientations, rows 2i (as is) and 2i + 1 (mirrored); p = (p_id + p_mir o mirror) * 0.5, v likewise.
#pragma once
#include <cassert>
#include "ccx_device.cuh"

// bounds of the mirrored indices, checked in a debug build (CCX_NVCC_EXTRA=-DCCX_DEBUG_BOUNDS): every mirrored cell lies in
// [0, 49) and every mirrored policy index in [0, 294), because both maps are involutions of those ranges
#ifdef CCX_DEBUG_BOUNDS
#define SYM_BOUND(c) assert(c)
#else
#define SYM_BOUND(c) ((void)0)
#endif

enum { SYM_OFF = 0, SYM_RANDOM = 1, SYM_MEAN = 2 };
#define SYM_COUNTER 0x53594Du              // "SYM": second counter word of the orientation draw

// net rows per evaluated position
template <int SYM> struct SymRows { static constexpr int value = SYM == SYM_MEAN ? 2 : 1; };

// the mirror of board cell r*7 + c and of policy index id*49 + r*7 + c (both involutions)
__device__ __forceinline__ int sym_mirror_cell(int rc) { const int r = rc / 7, c = rc - 7 * r; return (6 - c) * 7 + (6 - r); }
__device__ __forceinline__ int sym_mirror_action(int a) { const int id = a / 49; return id * 49 + sym_mirror_cell(a - 49 * id); }

// SYM_RANDOM's orientation of the position with state words OCC1, OCC2, META: h(s) = fold32(OCC1 * 0x9E3779B97F4A7C15 +
// OCC2 * 0xC2B2AE3D27D4EB4F + (META & 0xFFFFFFFFFFFF)), as the tie rule's root hash; true = evaluate mirrored
__device__ __forceinline__ bool sym_mirrored(u32 k0, u32 k1, u64 occ1, u64 occ2, u64 meta)
{
    const u64 z = occ1 * 0x9E3779B97F4A7C15ULL + occ2 * 0xC2B2AE3D27D4EB4FULL + (meta & 0x0000FFFFFFFFFFFFULL);
    return philox4x32_10(k0, k1, (u32)(z >> 32) ^ (u32)z, SYM_COUNTER, 0u, 0u).x & 1u;
}

__device__ __forceinline__ bool sym_mirrored(u32 k0, u32 k1, const Game &g)
{
    const bool p2 = (g.meta >> 48) & 1;
    return sym_mirrored(k0, k1, p2 ? g.occ_op : g.occ_me, p2 ? g.occ_me : g.occ_op, g.meta);
}

// utils.to_model_input of g into dst[343], cells mirrored when `mir` (staged in sp[352]: zero, scatter the 36 labels, copy out)
__device__ __forceinline__ void encode_planes(const Game &g, int lane, bool mir, uint8_t *__restrict__ sp, uint8_t *__restrict__ dst)
{
    for (int i = lane; i < 88; i += 32) reinterpret_cast<uint32_t *>(sp)[i] = 0u;
    __syncwarp();
    const int plies = (int)((g.meta >> 32) & 0xFFFF);
    const u64 cur0 = g.cells_me, opp0 = g.cells_op;
    const u64 opp1 = undo_in_cells(opp0, (int)(g.meta & 0xFF), (int)((g.meta >> 8) & 0xFF));
    const u64 cur2 = undo_in_cells(cur0, (int)((g.meta >> 16) & 0xFF), (int)((g.meta >> 24) & 0xFF));
    for (int e = lane; e < 36; e += 32) {
        int hs = e / 12, side = (e / 6) & 1, id = e % 6;
        if (hs > plies) continue;
        u64 cells = side ? (hs >= 1 ? opp1 : opp0) : (hs >= 2 ? cur2 : cur0);
        int c = (int)((cells >> (8 * id)) & 0xFF);
        if (c < 55 && (c & 7) < 7) {
            const int r = c >> 3, col = c & 7;
            const int cell = mir ? (6 - col) * 7 + (6 - r) : r * 7 + col;
            SYM_BOUND(cell >= 0 && cell < 49);
            sp[cell * 7 + 2 * hs + side] = (uint8_t)(id + 1);
        }
    }
    if ((g.meta >> 48) & 1)
        for (int c = lane; c < 49; c += 32) sp[c * 7 + 6] = 1;                    // utils.py:157-158
    __syncwarp();
    for (int i = lane; i < 343; i += 32) dst[i] = sp[i];
}

// the net input rows of one position in SYM's layout, dst = planes + position * SymRows<SYM> * 343
template <int SYM>
__device__ __forceinline__ void sym_encode(const Game &g, int lane, u32 k0, u32 k1, uint8_t *__restrict__ sp, uint8_t *__restrict__ dst)
{
    if constexpr (SYM == SYM_MEAN) {
        encode_planes(g, lane, false, sp, dst);
        __syncwarp();                                                             // sp is staged again
        encode_planes(g, lane, true, sp, dst + 343);
    } else {
        encode_planes(g, lane, SYM == SYM_RANDOM && sym_mirrored(k0, k1, g), sp, dst);
    }
}

// utils.softmax in float64 over the 294 logits of one row (model.py:21-24, utils.py:187-192): x[j] = exp(l[i] - max l) for
// i = lane + 32 j (0 past the end); returns the warp's sum
__device__ __forceinline__ double sym_softmax_row(int lane, const float *__restrict__ lg, double (&x)[10])
{
    double mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < 10; j++) {
        int i = lane + 32 * j;
        x[j] = i < 294 ? (double)lg[i] : -INFINITY;
        mx = fmax(mx, x[j]);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) mx = fmax(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, off));
    double sum = 0.0;
#pragma unroll
    for (int j = 0; j < 10; j++) { x[j] = (lane + 32 * j) < 294 ? exp(x[j] - mx) : 0.0; sum += x[j]; }
#pragma unroll
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, off);
    return sum;
}

// priors p[294] of one position from its net rows lg (SymRows<SYM> rows of 294 logits); `mir` = SYM_RANDOM's orientation.
// SYM_OFF: p = softmax(lg); SYM_RANDOM: p[mirror(i)] = softmax(lg)[i] when mirrored; SYM_MEAN: p[a] = (p_id[a] + p_mir[mirror(a)]) * 0.5.
// The caller synchronises the warp before p is read by other lanes.
template <int SYM>
__device__ __forceinline__ void sym_priors(int lane, const float *__restrict__ lg, bool mir, double *__restrict__ p)
{
    double x[10];
    double sum = sym_softmax_row(lane, lg, x);
#pragma unroll
    for (int j = 0; j < 10; j++) {
        const int i = lane + 32 * j;
        if (i < 294) {
            const int a = SYM == SYM_RANDOM && mir ? sym_mirror_action(i) : i;
            SYM_BOUND(a >= 0 && a < 294);
            p[a] = x[j] / sum;
        }
    }
    if constexpr (SYM == SYM_MEAN) {
        __syncwarp();
        sum = sym_softmax_row(lane, lg + 294, x);
#pragma unroll
        for (int j = 0; j < 10; j++) {
            const int i = lane + 32 * j;      // index in the mirrored frame; each a is written by one (lane, j)
            if (i < 294) {
                const int a = sym_mirror_action(i);
                SYM_BOUND(a >= 0 && a < 294);
                p[a] = __dmul_rn(__dadd_rn(p[a], x[j] / sum), 0.5);
            }
        }
    }
}

// value of one position from its net rows' values (SymRows<SYM> floats)
template <int SYM>
__device__ __forceinline__ double sym_value(const float *__restrict__ val)
{
    if constexpr (SYM == SYM_MEAN) return __dmul_rn(__dadd_rn((double)val[0], (double)val[1]), 0.5);
    else return (double)val[0];
}
