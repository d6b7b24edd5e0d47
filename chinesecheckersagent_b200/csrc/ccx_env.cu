// ccx_env.cu — env kernels (movegen / apply / win / random + greedy stepping / plane encoder) and the
// handle part of the C-ABI declared in include/ccx.h.  Hand-written for sm_100a; one thread per game,
// SoA words so that a warp's loads and stores are 256-byte contiguous.
#include <cuda_bf16.h>
#include <new>
#include <cstdlib>
#include "ccx_device.cuh"
#include "ccx_internal.h"

#ifndef CCX_GREEDY_DEFAULT_VARIANT
#define CCX_GREEDY_DEFAULT_VARIANT 1      // k_play_greedy_tri<448, 2>: 6.78e9 plies/s against 4.57e9 for k_play_greedy at 131,072 games (profiles/r02c_greedy_variants.log)
#endif
#define ENV_THREADS 64      // 1024 blocks of 2 warps for 65,536 games: 6.9 blocks per SM (148 SMs), 98.8 % balanced
#define ENC_THREADS 128

// --------------------------------------------------------------------------------------------------
// state load / store (side-to-move relative)

__device__ __forceinline__ Game load_game(const u64 *__restrict__ st, int64_t n, int64_t i)
{
    u64 occ1 = st[0 * n + i], occ2 = st[1 * n + i], c1 = st[2 * n + i], c2 = st[3 * n + i];
    Game g;
    g.meta = st[4 * n + i];
    bool p2 = (g.meta >> 48) & 1;
    g.occ_me = p2 ? occ2 : occ1; g.occ_op = p2 ? occ1 : occ2;
    g.cells_me = p2 ? c2 : c1;   g.cells_op = p2 ? c1 : c2;
    return g;
}

__device__ __forceinline__ void store_game(u64 *__restrict__ st, int64_t n, int64_t i, const Game &g)
{
    bool p2 = (g.meta >> 48) & 1;
    st[0 * n + i] = p2 ? g.occ_op : g.occ_me;
    st[1 * n + i] = p2 ? g.occ_me : g.occ_op;
    st[2 * n + i] = p2 ? g.cells_op : g.cells_me;
    st[3 * n + i] = p2 ? g.cells_me : g.cells_op;
    st[4 * n + i] = g.meta;
}

// ray-jump table: built once per handle in global memory, staged into shared memory by every block
__global__ void k_build_jump_table(uint8_t *T) { build_jump_table(T, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x); }

#define LOAD_JUMP_TABLE(sT, gT)                                                                   \
    __shared__ __align__(16) uint8_t sT[CCX_JT_BYTES];                                            \
    for (int q__ = threadIdx.x; q__ < CCX_JT_BYTES / 16; q__ += blockDim.x)                        \
        reinterpret_cast<uint4 *>(sT)[q__] = reinterpret_cast<const uint4 *>(gT)[q__];             \
    __syncthreads();

// --------------------------------------------------------------------------------------------------
// K0 reset  (board.py:10-57, 61-85)

__global__ void __launch_bounds__(ENV_THREADS)
k_reset(u64 *__restrict__ st, int64_t n, int mode, u32 k0, u32 k1, int64_t gid0)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 occ[2] = {CCX_START_OCC1, CCX_START_OCC2}, cells[2] = {CCX_START_CELLS1, CCX_START_CELLS2};
    if (mode == CCX_RESET_RANDOMISED) {
        // 12 draws without replacement: the k-th free cell, k = mulhi(rnd, #free)  (board.py:69)
        u64 gid = (u64)(gid0 + i);
        u64 taken = 0;
        occ[0] = occ[1] = cells[0] = cells[1] = 0;
#pragma unroll
        for (int q = 0; q < 3; q++) {
            Philox4 r = philox4x32_10(k0, k1, (u32)q, 2u, (u32)gid, (u32)(gid >> 32));
            u32 rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                int idx = q * 4 + j;
                u32 k = __umulhi(rr[j], (u32)(49 - idx));
                int cell = select64(~taken & CCX_VALID, k);
                taken |= 1ULL << cell;
                int pl = idx / 6, id = idx % 6;
                occ[pl] |= 1ULL << cell;
                cells[pl] |= (u64)cell << (8 * id);
            }
        }
    }
    st[0 * n + i] = occ[0]; st[1 * n + i] = occ[1];
    st[2 * n + i] = cells[0]; st[3 * n + i] = cells[1];
    st[4 * n + i] = CCX_START_META;
    st[5 * n + i] = CCX_HIST_EMPTY; st[6 * n + i] = CCX_HIST_EMPTY;
    st[7 * n + i] = 0;
}

// --------------------------------------------------------------------------------------------------
// K1 movegen  (board.py:139-222)

__global__ void __launch_bounds__(ENV_THREADS)
k_movegen(const u64 *__restrict__ st, int64_t n, u64 *__restrict__ masks, const uint8_t *__restrict__ jt)
{
    LOAD_JUMP_TABLE(sT, jt)
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Game g = load_game(st, n, i);
    u64 dest[6];
    movegen_rays(g.occ_me | g.occ_op, g.cells_me, dest, sT);
#pragma unroll
    for (int k = 0; k < 6; k++) masks[k * n + i] = dest[k];
}

// --------------------------------------------------------------------------------------------------
// K2/K3 apply + win  (board.py:226-250, 89-111)

__global__ void __launch_bounds__(ENV_THREADS)
k_apply(u64 *__restrict__ st, int64_t n, const uint8_t *__restrict__ from, const uint8_t *__restrict__ to,
        uint8_t *__restrict__ winner)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Game g = load_game(st, n, i);
    int f = from[i], t = to[i];
    int id = 0;
#pragma unroll
    for (int k = 5; k >= 0; k--) if (((g.cells_me >> (8 * k)) & 0xFF) == (u64)f) id = k;   // board.py:235-238
    apply_move(g, id, f, t);
    store_game(st, n, i, g);
    u64 lo = st[5 * n + i], hi = st[6 * n + i];
    push_hist(lo, hi, t);
    st[5 * n + i] = lo; st[6 * n + i] = hi;
    winner[i] = (uint8_t)winner_of(g);
}

__global__ void __launch_bounds__(ENV_THREADS)
k_info(const u64 *__restrict__ st, int64_t n, int16_t *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 occ1 = st[0 * n + i], occ2 = st[1 * n + i], c1 = st[2 * n + i], c2 = st[3 * n + i];
    int d1 = 70, d2 = -14;                                     // config.py:13-14, board.py:270-288
#pragma unroll
    for (int k = 0; k < 6; k++) {
        d1 -= level_of((int)((c1 >> (8 * k)) & 0xFF)) + 1;
        d2 += level_of((int)((c2 >> (8 * k)) & 0xFF)) + 1;
    }
    out[i * 5 + 0] = (int16_t)check_win(occ1, occ2);
    out[i * 5 + 1] = (int16_t)__popcll(occ1 & CCX_TARGET_P1);  // board.py:254-266
    out[i * 5 + 2] = (int16_t)__popcll(occ2 & CCX_TARGET_P2);
    out[i * 5 + 3] = (int16_t)d1;
    out[i * 5 + 4] = (int16_t)d2;
}

// --------------------------------------------------------------------------------------------------
// fused random-legal env step  (selfplay.py:83-104 + board.py:226-250 + board.py:89-111)

// ray-jump table lookups and per-cell constants of the three-layout kernels, staged into ONE static shared array, so that
// all hot loads are [register + one uniform base + constant] (with separate arrays ptxas re-derives the extra bases from
// SR_CgaCtaId inside the loops).  SEL: the array also holds the rank table of select64_step (CCX_SEL7_BYTES more).
#define CCX_TRI_SMEM_BYTES (CCX_JT3_BYTES + 5 * 64 * 8)
template <int TPB, bool SEL = false>
__device__ __forceinline__ TriTables tri_tables_load(uint8_t *sAll, const uint8_t *__restrict__ jt3)
{
    u64 *sNB = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES), *sCI = sNB + 64, *sO = sNB + 128, *sOT = sNB + 192, *sOD = sNB + 256;
    u32 *sSel = SEL ? reinterpret_cast<u32 *>(sAll + CCX_TRI_SMEM_BYTES) : nullptr;
    for (int q = threadIdx.x; q < CCX_JT3_BYTES / 16; q += TPB) reinterpret_cast<uint4 *>(sAll)[q] = reinterpret_cast<const uint4 *>(jt3)[q];
    for (int q = threadIdx.x; q < 64; q += TPB) {
        const bool on = (CCX_VALID >> q) & 1;
        sNB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
        sCI[q] = on ? tri_cell_info(q) : 0ULL;
        sO[q] = 1ULL << q;
        sOT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
        sOD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
    }
    if (SEL)
        for (int q = threadIdx.x; q < 128; q += TPB) sSel[q] = sel7_entry((u32)q);
    __syncthreads();
    TriTables t = {sAll, sNB, sCI, sO, sOT, sOD, sSel};
    return t;
}

// The one-wave carry kernel's tables in dynamic shared memory (CCX_WIDE_SMEM_BYTES, 194.5 KB: one block per SM): the wide
// answer tables (build_jump_table_wide) instead of build_jump_table3's and tri_cell_info, then sNB / sO / sOT / sOD and the
// rank table.  The 192 KB copy keeps four 16-byte loads per lane in flight.
#define CCX_WIDE_SMEM_BYTES (CCX_JTW_BYTES + 4 * 64 * 8 + CCX_SEL7_BYTES)
template <int TPB>
__device__ __forceinline__ TriTables wide_tables_load(uint8_t *s, const u64 *__restrict__ jtw)
{
    u64 *sW = reinterpret_cast<u64 *>(s), *sNB = sW + 3 * 128 * 64, *sO = sNB + 64, *sOT = sNB + 128, *sOD = sNB + 192;
    u32 *sSel = reinterpret_cast<u32 *>(sNB + 256);
    constexpr int N = CCX_JTW_BYTES / 16, U = 4;
    const uint4 *src = reinterpret_cast<const uint4 *>(jtw);
    uint4 *dst = reinterpret_cast<uint4 *>(s);
    for (int q = threadIdx.x; q < N; q += U * TPB) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; u++) if (q + u * TPB < N) v[u] = src[q + u * TPB];
#pragma unroll
        for (int u = 0; u < U; u++) if (q + u * TPB < N) dst[q + u * TPB] = v[u];
    }
    for (int q = threadIdx.x; q < 64; q += TPB) {
        const bool on = (CCX_VALID >> q) & 1;
        sNB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
        sO[q] = 1ULL << q;
        sOT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
        sOD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
    }
    for (int q = threadIdx.x; q < 128; q += TPB) sSel[q] = sel7_entry((u32)q);
    __syncthreads();
    TriTables t = {nullptr, sNB, nullptr, sO, sOT, sOD, sSel, sW};
    return t;
}

// --------------------------------------------------------------------------------------------------
// fused random-legal env step  (selfplay.py:83-104 + board.py:226-250 + board.py:89-111)
//
// Pick first (pick_random_first, ccx_device.cuh): the random choice needs only which checkers can move and the full
// destination set of the one it picks, so a ply runs the walk test of all six checkers (one set-parallel pass), one
// expansion for the rare checker without an empty neighbour, Philox, the pick, and the jump flood fill of the picked checker
// alone: ~3.5 expanded cells per game-ply instead of ~21 for all six closures.  One game per lane, its state in registers
// for all plies; a warp runs the fill as long as its longest lane (~10 iterations per warp-ply).  The occupancy is also kept
// column- and diagonal-major (a move flips two bits in each copy) for expand_cell_tri.  The tables are static (47.5 KB), so
// one 448-lane block per SM covers 148 x 448 = 66,304 games in one wave; larger batches run two blocks per SM (MINB = 2,
// at most 72 registers).  Same per-game Philox counters and moves as every earlier step kernel.
// TRACE: rows carry all six destination sets, so traced games also run movegen_tri for the row; their move still comes
// from the pick-first path, which the trace parity test therefore checks ply by ply against the oracle.
// Tried and dropped with the earlier all-six-closures kernels (B200, 65,536 games; the lessons carry over): two lanes per
// game, three checkers each (3.90e9 against 4.35e9 steps/s: the pair votes and waits cost more than the extra warps hide);
// two games or two checker streams per lane for instruction-level parallelism (3.93e9, and 4.11 / 4.16 ms against 3.39 ms:
// the dummy expansions of a stream that has run dry outweigh the overlapped latencies); fewer games per warp (28 / 24 / 22 /
// 16 of 32 lanes: 4.43e9 / 3.77e9 / 3.25e9 / 2.84e9 against 4.42e9: the rate follows warp instructions issued, not occupancy).
template <bool TRACE, int TPB, int MINB>
__global__ void __launch_bounds__(TPB, MINB, 1)   // cluster size bound 1: the shared-window base stays in a uniform register across the loop
k_step_random_pick(u64 *__restrict__ st, int64_t n, int64_t gid0, u32 k0, u32 k1, u32 step0, int plies,
                   u64 *__restrict__ wins, u64 *__restrict__ trace, int64_t trace_games, const uint8_t *__restrict__ jt3)
{
    __shared__ __align__(16) uint8_t sAll[CCX_JT3_BYTES + 5 * 64 * 8];
    const TriTables T = tri_tables_load<TPB>(sAll, jt3);
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;                       // no warp-wide votes below: lanes past the end may leave
    Game g = load_game(st, n, i);
    const u64 gid = (u64)(gid0 + i);
    u32 w1 = 0, w2 = 0;
    u64 occT_all, occD_all;
    tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all);
    for (int t = 0; t < plies; t++) {
        u64 *row = nullptr;
        if (TRACE && i < trace_games) {
            row = trace + ((int64_t)t * trace_games + i) * CCX_TRACE_WORDS;
            u64 dest[6];
            movegen_tri(g.occ_me | g.occ_op, occT_all, occD_all, g.cells_me, dest, T);
            bool p2 = (g.meta >> 48) & 1;
            row[0] = p2 ? g.occ_op : g.occ_me; row[1] = p2 ? g.occ_me : g.occ_op;
            row[2] = p2 ? g.cells_op : g.cells_me; row[3] = p2 ? g.cells_me : g.cells_op;
            row[4] = g.meta & 0x00FFFFFFFFFFFFFFULL;
#pragma unroll
            for (int q = 0; q < 6; q++) row[5 + q] = dest[q];
            row[11] = 0xFFULL | (0xFFULL << 8) | (0xFFULL << 24);
        }
        Philox4 rnd = philox4x32_10(k0, k1, step0 + (u32)t, 0u, (u32)gid, (u32)(gid >> 32));
        int from, to;
        const int pid = pick_random_first(g, occT_all, occD_all, rnd.x, rnd.y, T, from, to);
        if (pid < 0) continue;                // no checker can move: the ply passes, as in the oracle
        apply_move(g, pid, from, to);
        occT_all ^= T.sOT[from] | T.sOT[to];
        occD_all ^= T.sOD[from] | T.sOD[to];
        const int win = winner_of(g);
        if (TRACE && row) row[11] = (u64)from | ((u64)to << 8) | ((u64)win << 16) | ((u64)pid << 24);
        if (win) { w1 += win == 1; w2 += win == 2; reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
    }
    store_game(st, n, i, g);
    if (w1) atomicAdd(&wins[0], (u64)w1);
    if (w2) atomicAdd(&wins[1], (u64)w2);
}

// k_step_random_pick with the flood fill bounded per round: a lane runs at most K fill steps, then the warp goes on, and a
// lane whose closure needs more carries its fill (and the ply's checker, origin and r1) into the next round.  A round is:
// lanes whose fill is done finish their ply (destination, apply, win, and the next ply's Philox words) and start their next
// one (walk test, pick, fill start), then every lane runs up to K fill steps.  So lanes may be on different plies, and a warp
// waits for its longest lane's fill only up to K steps at a time instead of for the whole closure; the per-ply path of the
// ready lanes runs about once per round.  A lane leaves once it has played all its plies.  A game's Philox counters, moves and
// results are those of k_step_random_pick; only the interleaving of the lanes differs.
// The per-ply path (carry_ply_start / carry_ply_to, ccx_device.cuh) makes k_step_random_pick's choice with shorter chains:
// the checker picked speculatively as if all six had a walk (the exact pick by the rank table only when one has none), the
// destination by select64_step, the destination set gathered in the fill's `reach`, the occupancy words rebuilt from the
// fill's, and the Philox rounds overlapping the previous ply's finish.
// The fill (fill_step_carry / carry_fill_start) has a shorter dependent chain than fill_step: the per-cell constants come
// from the cell by ALU instructions (carry_cell) instead of a tri_cell_info load, the top bit from two FLOs in parallel, and
// the origin's expansion, which needs no FLO and no mover-free occupancy, runs in the ply start, so the K steps of a round
// begin at the ply's second.  In the one-wave launch (MINB = 1) the expansions run over the wide answer tables
// (build_jump_table_wide, 192 KB of dynamic shared memory): three PRMTs, three IMAD addresses, three LDS.64 and the ORs, with no
// shift of an answer, 37 SASS instructions per fill step against 52; TRACE rows there run movegen_tri over the same tables.
// Two blocks per SM have no room for them and keep build_jump_table3's (profiles/r05_*).  Before the wide tables: SASS (sm_100a, <false, 448, 1,
// 5>, loop head to the first fill step without the win reset and the no-walk loop): 297 instructions per round against 262
// before (the origin's expansion moved in), a fill step 52 against 50 (FLO to FLO), one shared-memory load per step on the
// dependent chain instead of two.  Measured (B200, profiles/r03d_*): 0.545 -> 0.528 ms at 65,536 games (K = 5); with K = 5
// the extra instructions cost 0.4 % at 1 M games (28 warps per SM, closer to issue-bound), where K = 4 is 1.0 % faster than
// K = 5, so the launch runs K = 5 in one wave and K = 4 beyond: 0.935 -> 0.914 ms at 131,072 games, 6.864 -> 6.817 ms at 1 M.
template <bool TRACE, int TPB, int MINB, int K>
__global__ void __launch_bounds__(TPB, MINB, 1)
k_step_random_carry(u64 *__restrict__ st, int64_t n, int64_t gid0, u32 k0, u32 k1, u32 step0, int plies,
                    u64 *__restrict__ wins, u64 *__restrict__ trace, int64_t trace_games, const uint8_t *__restrict__ jt3,
                    const u64 *__restrict__ jtw)
{
    // One block per SM (the one-wave launch) has the room for the wide answer tables (CCX_WIDE_SMEM_BYTES of dynamic shared
    // memory); two per SM run on build_jump_table3's, in the static array.
    constexpr bool WIDE = MINB == 1;
    extern __shared__ __align__(16) u64 sDyn[];
    __shared__ __align__(16) uint8_t sAll[WIDE ? 16 : CCX_TRI_SMEM_BYTES + CCX_SEL7_BYTES];     // 49,152 B: the static limit
    const TriTables T = WIDE ? wide_tables_load<TPB>(reinterpret_cast<uint8_t *>(sDyn), jtw) : tri_tables_load<TPB, true>(sAll, jt3);
    const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    if (i >= n) return;                       // no warp-wide votes below: lanes past the end may leave
    Game g = load_game(st, n, i);
    const u64 gid = (u64)(gid0 + i);
    u32 w1 = 0, w2 = 0;
    // Before the first ply f.occT / f.occD hold the whole occupancy in the T / D layouts (with f.o = 0); from then on they hold
    // it without the mover of the ply, and the next occupancy follows from them and `to`.  So the full-board words are not
    // carried through the fill.
    JumpFill f = {0, 0, 0, 0, 0, 0};
    tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, f.occT, f.occD);
    int t = 0, id = -1, from = 0;             // id >= 0: ply t has picked checker id (on cell from); its fill runs or is done
    // Philox words of the next ply to start.  A ply's words are drawn while the ply before it finishes, so the ten dependent
    // rounds overlap that ply's destination select and move instead of preceding the next pick.
    Philox4 rnd = philox4x32_10(k0, k1, step0, 0u, (u32)gid, (u32)(gid >> 32));
    u32 r1 = 0;
    for (;;) {
        if (!f.todo) {
            u64 occT_all = f.occT, occD_all = f.occD;
            if (id >= 0) {                    // the fill of ply t is done: finish the ply
                rnd = philox4x32_10(k0, k1, step0 + (u32)t + 1u, 0u, (u32)gid, (u32)(gid >> 32));
                const int to = carry_ply_to(f, r1, T);
                apply_move(g, id, from, to);
                occT_all |= T.sOT[to];         // `to` was empty
                occD_all |= T.sOD[to];
#ifdef __CUDA_ARCH__
                asm volatile("" ::"r"(rnd.x), "r"(rnd.y));     // keeps the draw in this block (the compiler would sink it past the win branch)
#endif
                const int win = winner_of(g);
                if (TRACE && i < trace_games)
                    trace[((int64_t)t * trace_games + i) * CCX_TRACE_WORDS + 11] = (u64)from | ((u64)to << 8) | ((u64)win << 16) | ((u64)id << 24);
                if (win) { w1 += win == 1; w2 += win == 2; reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
                t++;
                id = -1;
            }
            for (; t < plies; t++) {          // start ply t; a ply in which no checker can move passes, as in the oracle
                if (TRACE && i < trace_games) {
                    u64 *row = trace + ((int64_t)t * trace_games + i) * CCX_TRACE_WORDS;
                    u64 dest[6];
                    movegen_tri<WIDE>(g.occ_me | g.occ_op, occT_all, occD_all, g.cells_me, dest, T);
                    bool p2 = (g.meta >> 48) & 1;
                    row[0] = p2 ? g.occ_op : g.occ_me; row[1] = p2 ? g.occ_me : g.occ_op;
                    row[2] = p2 ? g.cells_op : g.cells_me; row[3] = p2 ? g.cells_me : g.cells_op;
                    row[4] = g.meta & 0x00FFFFFFFFFFFFFFULL;
#pragma unroll
                    for (int q = 0; q < 6; q++) row[5 + q] = dest[q];
                    row[11] = 0xFFULL | (0xFFULL << 8) | (0xFFULL << 24);
                }
                r1 = rnd.y;
                id = carry_ply_start<WIDE>(g, occT_all, occD_all, rnd.x, T, from, f);
                if (id >= 0) break;
                rnd = philox4x32_10(k0, k1, step0 + (u32)t + 1u, 0u, (u32)gid, (u32)(gid >> 32));
            }
            if (id < 0) break;                // all plies played
        }
        // every lane still here has a fill, which may be done already (carry_ply_start takes its first step).  Unrolled: a
        // loop counter costs 4 of the ~50 instructions of a fill step (0.620 against 0.606 ms at K = 5, 65,536 games)
#pragma unroll
        for (int k = 0; k < K; k++) { if (!f.todo) break; fill_step_carry(f, carry_tables<WIDE>(T)); }
    }
    store_game(st, n, i, g);
    if (w1) atomicAdd(&wins[0], (u64)w1);
    if (w2) atomicAdd(&wins[1], (u64)w2);
}

// --------------------------------------------------------------------------------------------------
// Work-queue step kernel (the default before k_step_random_pick; CCX_STEP_VARIANT=9 runs it): a warp owns 32 games and steps them ply by ply TOGETHER; within a ply the
// 32 x 6 checker flood fills are work items that the lanes take from a warp-wide queue (a ballot + popc hands out the next
// indices), so a lane that finishes a short closure continues with another game's checker instead of waiting: the ply costs
// ~(total expansions) / 32 iterations instead of the longest lane's, and the pick / apply / win / Philox tail runs once per
// ply with all 32 lanes.  Same three-layout expansion and tables as k_step_random_pick; bit-identical results.
// PRE: the owner lane of a game writes the four words of each of its six items (mover bit, occupancy without the mover in the
// three layouts) to shared memory at the start of the ply, with all 32 lanes active, instead of every lane deriving them when it
// takes an item (a divergent block that runs for ~7 lanes in nearly every iteration).  Costs 24 KB more shared memory per 448 lanes.
template <bool TRACE, int TPB, int MINB, bool PRE>
__global__ void __launch_bounds__(TPB, MINB, 1)
k_step_random_wq(u64 *__restrict__ st, int64_t n, int64_t gid0, u32 k0, u32 k1, u32 step0, int plies,
                 u64 *__restrict__ wins, u64 *__restrict__ trace, int64_t trace_games, const uint8_t *__restrict__ jt3)
{
    extern __shared__ __align__(16) u64 sDyn[];                       // per warp: [6][32] jump closures, then [4][32] game words of the ply
    __shared__ __align__(16) uint8_t sAll[CCX_JT3_BYTES + 5 * 64 * 8];
    const uint8_t *sT = sAll;
    u64 *sNB = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES);
    u64 *sCI = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES + 512);
    u64 *sO = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES + 1024);
    u64 *sOT = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES + 1536);
    u64 *sOD = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES + 2048);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int q = tid; q < CCX_JT3_BYTES / 16; q += TPB) reinterpret_cast<uint4 *>(sAll)[q] = reinterpret_cast<const uint4 *>(jt3)[q];
    for (int q = tid; q < 64; q += TPB) {
        const bool on = (CCX_VALID >> q) & 1;
        sNB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
        sCI[q] = on ? tri_cell_info(q) : 0ULL;
        sO[q] = 1ULL << q;
        sOT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
        sOD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
    }
    __syncthreads();
    constexpr int WARP_WORDS = PRE ? (6 + 4 * 6) * 32 : 10 * 32;
    u64 *sD = sDyn + warp * WARP_WORDS;         // [6][32]
    u64 *sG = sD + 6 * 32;                      // !PRE: [4][32] occ_all, occT_all, occD_all, cells_me of the warp's 32 games
                                                //  PRE: [4][192] per item (idx = checker * 32 + game): o, occ, occT, occD
    const int64_t i = (int64_t)blockIdx.x * TPB + tid;
    const bool act = i < n;
    Game g = load_game(st, n, act ? i : 0);
    if (!act) reset_start(g);                   // lanes past the end play a dummy game that is never stored
    const u64 gid = (u64)(gid0 + i);
    u32 w1 = 0, w2 = 0;
    u64 occT_all, occD_all;
    tri_build(g.cells_me, g.cells_op, sOT, sOD, occT_all, occD_all);
    const unsigned lt_mask = (1u << lane) - 1u;
    for (int t = 0; t < plies; t++) {
        const u64 occ_all = g.occ_me | g.occ_op;
        if (PRE) {
#pragma unroll
            for (int q = 0; q < 6; q++) {
                const int cell = (int)((g.cells_me >> (8 * q)) & 0x3F);
                const u64 oq = 1ULL << cell;      // a shift, not sO[cell]: the shared-memory data pipe is this kernel's busiest unit (78 %)
                sG[0 * 192 + q * 32 + lane] = oq;
                sG[1 * 192 + q * 32 + lane] = occ_all & ~oq;
                sG[2 * 192 + q * 32 + lane] = occT_all & ~sOT[cell];
                sG[3 * 192 + q * 32 + lane] = occD_all & ~sOD[cell];
            }
        } else {
            sG[0 * 32 + lane] = occ_all; sG[1 * 32 + lane] = occT_all; sG[2 * 32 + lane] = occD_all; sG[3 * 32 + lane] = g.cells_me;
        }
        __syncwarp();
        // ---- the ply's 192 flood fills from the warp's queue: item idx = checker (idx >> 5) of game (idx & 31)
        int next = 0, state = 0, gi = 0, k = 0;          // state: 0 wants an item, 1 working, 2 queue empty
        int working = 32;                                // lanes in state 0 or 1 (warp-uniform): the loop ends when it reaches 0
        u64 o = 0, occ = 0, occT = 0, occD = 0, todo = 0, reach = 0;
        for (;;) {
            const unsigned want = __ballot_sync(0xFFFFFFFFu, state == 0);      // the one vote per iteration
            if (want) {
                const int idx = next + __popc(want & lt_mask);
                const int asked = __popc(want), left = 192 - next;
                working -= asked > left ? asked - (left > 0 ? left : 0) : 0;      // lanes that find the queue empty retire
                next += asked;
                if (state == 0) {
                    if (idx < 192) {
                        if (PRE) {
                            gi = idx;                     // the parking slot sD[checker * 32 + game] is the item index itself
                            o = sG[0 * 192 + idx]; occ = sG[1 * 192 + idx]; occT = sG[2 * 192 + idx]; occD = sG[3 * 192 + idx];
                        } else {
                            gi = idx & 31; k = idx >> 5;
                            const int cell = (int)((sG[3 * 32 + gi] >> (8 * k)) & 0x3F);
                            o = sO[cell];
                            occ = sG[0 * 32 + gi] & ~o; occT = sG[1 * 32 + gi] & ~sOT[cell]; occD = sG[2 * 32 + gi] & ~sOD[cell];
                        }
                        todo = o; reach = 0; state = 1;
                    } else state = 2;
                }
                if (working == 0) break;
            }
            if (state == 1) {
                const int c = 63 - __clzll((long long)todo);
                todo ^= PRE ? 1ULL << c : sO[c];
                const u64 nw = expand_cell_tri(c, occ, occT, occD, sT, sCI) & ~(reach | o);
                reach |= nw;
                todo |= nw;
                if (todo == 0) { sD[PRE ? gi : k * 32 + gi] = reach; state = 0; }
            }
        }
        __syncwarp();
        // ---- tail, all 32 lanes: destinations = empty neighbours | jump closure, pick, apply, win
        u64 dest[6];
#pragma unroll
        for (int q = 0; q < 6; q++) dest[q] = sD[q * 32 + lane] | (sNB[(g.cells_me >> (8 * q)) & 0x3F] & ~occ_all);
        u32 nonempty = 0;
#pragma unroll
        for (int q = 0; q < 6; q++) nonempty += dest[q] != 0;
        u64 *row = nullptr;
        if (TRACE && i < trace_games) {
            row = trace + ((int64_t)t * trace_games + i) * CCX_TRACE_WORDS;
            bool p2 = (g.meta >> 48) & 1;
            row[0] = p2 ? g.occ_op : g.occ_me; row[1] = p2 ? g.occ_me : g.occ_op;
            row[2] = p2 ? g.cells_op : g.cells_me; row[3] = p2 ? g.cells_me : g.cells_op;
            row[4] = g.meta & 0x00FFFFFFFFFFFFFFULL;
#pragma unroll
            for (int q = 0; q < 6; q++) row[5 + q] = dest[q];
            row[11] = 0xFFULL | (0xFFULL << 8) | (0xFFULL << 24);
        }
        if (nonempty) {
            Philox4 rnd = philox4x32_10(k0, k1, step0 + (u32)t, 0u, (u32)gid, (u32)(gid >> 32));
            int from, to;
            int pid = pick_random(g, dest, nonempty, rnd.x, rnd.y, from, to);
            apply_move(g, pid, from, to);
            occT_all ^= sOT[from] | sOT[to];
            occD_all ^= sOD[from] | sOD[to];
            int win = winner_of(g);
            if (TRACE && row) row[11] = (u64)from | ((u64)to << 8) | ((u64)win << 16) | ((u64)pid << 24);
            if (win) { w1 += win == 1; w2 += win == 2; reset_start(g); tri_build(g.cells_me, g.cells_op, sOT, sOD, occT_all, occD_all); }
        }
        __syncwarp();                             // sD / sG are rewritten by the next ply
    }
    if (!act) return;
    store_game(st, n, i, g);
    if (w1) atomicAdd(&wins[0], (u64)w1);
    if (w2) atomicAdd(&wins[1], (u64)w2);
}

// Tried and dropped (r02, second session): TWO queue slots per lane in k_step_random_wq<PRE> — the loop body expands one cell of each
// slot in one straight-line block (an idle slot expands cell 0 of stale words, masked), so that the two dependent chains
// (FLO -> LDS -> PRMT -> LDS -> shift -> mask) interleave.  Bit-identical, 91 registers, but 3.09 ms against 2.43 ms per 65,536 games x
// 256 plies (profiles/r02h_env_variants.log): the dummy expansions of the drain and the second item-take / park blocks cost more
// than the interleaving hides — the same outcome as two games per lane in the flat kernel (variants 2 / 3).
// Shared-memory traffic (ncu: l1tex__data_pipe_lsu_wavefronts_mem_shared at 78 % of peak, half of the 548 M wavefronts are bank
// conflicts of the lanes' random table reads) is what the queue loop saturates first.  Measured trades of loads against ALU work
// (profiles/r02h_env_variants.log): one-bit masks by shift instead of sO[] in the PRE stage AND in the loop 2.435 -> 2.375 ms (kept;
// either one alone: no change); a 32-bit per-cell table with computed row / column selectors: 2.404 ms;
// skipping the lookups of lines without another checker (predicated loads): 2.52 ms; BYTE answers for columns and diagonals (u8
// tables compressed from the 64-bit ones at block start, LDS.U8 over 32 banks instead of LDS.64 over 16 bank pairs, the scatter a
// 64-bit multiply + mask as in round 1): 2.537 ms — all bit-identical, all dropped: loads and ALU work are balanced where they are.

__global__ void k_build_jump_table3(uint8_t *T3) { build_jump_table3(T3, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x); }
__global__ void k_build_jump_table_wide(u64 *W, const uint8_t *T3) { build_jump_table_wide(W, T3, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x); }

// --------------------------------------------------------------------------------------------------
// K4 greedy  (player.py:99-121, board_utils.py:3-7)

__global__ void __launch_bounds__(ENV_THREADS)
k_greedy_candidates(const u64 *__restrict__ st, int64_t n, u64 *__restrict__ masks, const uint8_t *__restrict__ jt)
{
    LOAD_JUMP_TABLE(sT, jt)
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Game g = load_game(st, n, i);
    u64 dest[6], cand[6];
    movegen_rays(g.occ_me | g.occ_op, g.cells_me, dest, sT);
    greedy_candidates(g, dest, cand);
#pragma unroll
    for (int k = 0; k < 6; k++) masks[k * n + i] = cand[k];
}

// Game.start (game.py:58-100) with two GreedyPlayers
// Tried and dropped (r01f): a flattened per-lane state machine for this loop (each lane moves on to its next checker inside one
// loop, the greedy tail batched at 12 ready lanes) — same games bit for bit, 4.43e9 plies/s against 4.57e9 for this kernel: games of a warp end at different plies,
// so the warp runs as long as its longest game either way and the heavier greedy tail runs for fewer lanes per execution.
__global__ void __launch_bounds__(ENV_THREADS)
k_play_greedy(u64 *__restrict__ st, int64_t n, int64_t gid0, u32 k0, u32 k1, int max_plies,
              u64 *__restrict__ counters, const uint8_t *__restrict__ jt)
{
    LOAD_JUMP_TABLE(sT, jt)
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 played = 0, w1 = 0, w2 = 0, rep = 0;
    if (i < n) {
        Game g = load_game(st, n, i);
        u64 lo = st[5 * n + i], hi = st[6 * n + i];
        u64 gid = (u64)(gid0 + i);
        int status = (int)(g.meta >> 56);
        for (int t = 0; status == CCX_ST_RUNNING && t < max_plies; t++) {
            u64 dest[6], cand[6];
            movegen_rays(g.occ_me | g.occ_op, g.cells_me, dest, sT);
            int total = greedy_candidates(g, dest, cand);
            if (total == 0) { status = CCX_ST_NO_MOVES; break; }     // reference raises (player.py:113)
            u32 ply = (u32)((g.meta >> 32) & 0xFFFF);
            Philox4 r = philox4x32_10(k0, k1, ply, 1u, (u32)gid, (u32)(gid >> 32));
            int from, to;
            int id = pick_candidate(g, cand, total, r.x, from, to);   // player.py:121
            apply_move(g, id, from, to);                              // game.py:65
            push_hist(lo, hi, to);
            played++;
            int win = winner_of(g);
            if (win) { status = win; w1 += win == 1; w2 += win == 2; break; }     // game.py:70-71
            if (((g.meta >> 32) & 0xFFFF) >= 16 && repetition_stop(lo, hi)) { status = CCX_ST_REPETITION; rep++; }
        }
        g.meta = (g.meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)status << 56);
        store_game(st, n, i, g);
        st[5 * n + i] = lo; st[6 * n + i] = hi;
    }
    if (counters) {
        // warp-aggregated counters: one atomic per warp per counter
        for (int off = 16; off; off >>= 1) {
            played += __shfl_down_sync(0xFFFFFFFFu, played, off);
            w1 += __shfl_down_sync(0xFFFFFFFFu, w1, off);
            w2 += __shfl_down_sync(0xFFFFFFFFu, w2, off);
            rep += __shfl_down_sync(0xFFFFFFFFu, rep, off);
        }
        if ((threadIdx.x & 31) == 0) {
            if (played) atomicAdd(&counters[0], (u64)played);
            if (w1) atomicAdd(&counters[1], (u64)w1);
            if (w2) atomicAdd(&counters[2], (u64)w2);
            if (rep) atomicAdd(&counters[3], (u64)rep);
        }
    }
}

// Game.start with two GreedyPlayers, three-layout move generation (movegen_tri): same games bit for bit as k_play_greedy,
// ~20 % fewer instructions per ply.
template <int TPB, int MINB>
__global__ void __launch_bounds__(TPB, MINB, 1)
k_play_greedy_tri(u64 *__restrict__ st, int64_t n, int64_t gid0, u32 k0, u32 k1, int max_plies,
                  u64 *__restrict__ counters, const uint8_t *__restrict__ jt3)
{
    __shared__ __align__(16) uint8_t sAll[CCX_JT3_BYTES + 5 * 64 * 8];
    const TriTables T = tri_tables_load<TPB>(sAll, jt3);
    int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
    u32 played = 0, w1 = 0, w2 = 0, rep = 0;
    if (i < n) {
        Game g = load_game(st, n, i);
        u64 lo = st[5 * n + i], hi = st[6 * n + i];
        u64 gid = (u64)(gid0 + i);
        int status = (int)(g.meta >> 56);
        u64 occT_all, occD_all;
        tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all);
        for (int t = 0; status == CCX_ST_RUNNING && t < max_plies; t++) {
            u64 dest[6], cand[6];
            movegen_tri(g.occ_me | g.occ_op, occT_all, occD_all, g.cells_me, dest, T);
            int total = greedy_candidates(g, dest, cand);
            if (total == 0) { status = CCX_ST_NO_MOVES; break; }     // reference raises (player.py:113)
            u32 ply = (u32)((g.meta >> 32) & 0xFFFF);
            Philox4 r = philox4x32_10(k0, k1, ply, 1u, (u32)gid, (u32)(gid >> 32));
            int from, to;
            int id = pick_candidate(g, cand, total, r.x, from, to);   // player.py:121
            apply_move(g, id, from, to);                              // game.py:65
            occT_all ^= T.sOT[from] | T.sOT[to];
            occD_all ^= T.sOD[from] | T.sOD[to];
            push_hist(lo, hi, to);
            played++;
            int win = winner_of(g);
            if (win) { status = win; w1 += win == 1; w2 += win == 2; break; }     // game.py:70-71
            if (((g.meta >> 32) & 0xFFFF) >= 16 && repetition_stop(lo, hi)) { status = CCX_ST_REPETITION; rep++; }
        }
        g.meta = (g.meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)status << 56);
        store_game(st, n, i, g);
        st[5 * n + i] = lo; st[6 * n + i] = hi;
    }
    if (counters) {
        for (int off = 16; off; off >>= 1) {
            played += __shfl_down_sync(0xFFFFFFFFu, played, off);
            w1 += __shfl_down_sync(0xFFFFFFFFu, w1, off);
            w2 += __shfl_down_sync(0xFFFFFFFFu, w2, off);
            rep += __shfl_down_sync(0xFFFFFFFFu, rep, off);
        }
        if ((threadIdx.x & 31) == 0) {
            if (played) atomicAdd(&counters[0], (u64)played);
            if (w1) atomicAdd(&counters[1], (u64)w1);
            if (w2) atomicAdd(&counters[2], (u64)w2);
            if (rep) atomicAdd(&counters[3], (u64)rep);
        }
    }
}

// Tried and dropped (r02): Game.start as a warp work queue like k_step_random_wq (the warp's 32 games ply by ply, the flood fills of
// the games still running handed out from a warp-wide queue, one greedy tail per ply): same games bit for bit, but 0.996 ms per
// 131,072 games against 0.841 ms for k_play_greedy_tri — games end at different plies, so a ply-synchronous warp spends its last
// 20-30 plies on a handful of games at full per-ply overhead, and the 156 KB block leaves one block per SM.

// --------------------------------------------------------------------------------------------------
// K5 plane encoder  (utils.py:101-160): planes (2k, 2k+1) = id-labelled (mover, opponent) position k
// plies ago, k < min(plies, 2) + 1; plane 6 = 1 iff player 2 is to move.  Each block stages G games'
// (7,7,7) tensors in shared memory (scatter of 12 labels per history step) and streams them out with
// 16-byte stores, so HBM sees one contiguous G*343*sizeof(T) write per block.

template <typename T> __device__ __forceinline__ T enc_val(int v);
template <> __device__ __forceinline__ uint8_t enc_val<uint8_t>(int v) { return (uint8_t)v; }
template <> __device__ __forceinline__ float enc_val<float>(int v) { return (float)v; }
template <> __device__ __forceinline__ __nv_bfloat16 enc_val<__nv_bfloat16>(int v) { return __int2bfloat16_rn(v); }

template <typename T, int G>
__global__ void __launch_bounds__(ENC_THREADS)
k_encode(const u64 *__restrict__ st, int64_t n, T *__restrict__ out)
{
    extern __shared__ uint4 smem_u4[];
    T *tile = reinterpret_cast<T *>(smem_u4);
    constexpr int TILE_BYTES = G * 343 * (int)sizeof(T);
    static_assert(TILE_BYTES % 16 == 0, "tile must be a whole number of 16-byte vectors");
    int64_t g0 = (int64_t)blockIdx.x * G;
    int games = (int)min((int64_t)G, n - g0);
    for (int v = threadIdx.x; v < TILE_BYTES / 16; v += blockDim.x) smem_u4[v] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    for (int lg = threadIdx.x; lg < games; lg += blockDim.x) {
        int64_t i = g0 + lg;
        u64 c1 = st[2 * n + i], c2 = st[3 * n + i], meta = st[4 * n + i];
        bool p2 = (meta >> 48) & 1;
        u64 cur = p2 ? c2 : c1, opp = p2 ? c1 : c2;
        int plies = (int)((meta >> 32) & 0xFFFF);
        T *t = tile + lg * 343;
#pragma unroll
        for (int h = 0; h < 3; h++) {
            if (h == 1) { if (plies < 1) break; opp = undo_in_cells(opp, (int)(meta & 0xFF), (int)((meta >> 8) & 0xFF)); }
            if (h == 2) { if (plies < 2) break; cur = undo_in_cells(cur, (int)((meta >> 16) & 0xFF), (int)((meta >> 24) & 0xFF)); }
#pragma unroll
            for (int k = 0; k < 6; k++) {
                int a = (int)((cur >> (8 * k)) & 0xFF), b = (int)((opp >> (8 * k)) & 0xFF);
                // cells of a well-formed state are < 55 with column < 7; anything else is ignored, never written
                if (a < 55 && (a & 7) < 7) t[((a >> 3) * 7 + (a & 7)) * 7 + 2 * h] = enc_val<T>(k + 1);
                if (b < 55 && (b & 7) < 7) t[((b >> 3) * 7 + (b & 7)) * 7 + 2 * h + 1] = enc_val<T>(k + 1);
            }
        }
        if (p2)
            for (int c = 0; c < 49; c++) t[c * 7 + 6] = enc_val<T>(1);
    }
    __syncthreads();
    char *dst = reinterpret_cast<char *>(out) + g0 * 343 * (int64_t)sizeof(T);
    int bytes = games * 343 * (int)sizeof(T);
    int nvec = bytes / 16;       // block base offset is a multiple of 16 bytes because TILE_BYTES is
    uint4 *dst4 = reinterpret_cast<uint4 *>(dst);
    for (int v = threadIdx.x; v < nvec; v += blockDim.x) dst4[v] = smem_u4[v];
    const char *src = reinterpret_cast<const char *>(smem_u4);
    for (int b = nvec * 16 + threadIdx.x; b < bytes; b += blockDim.x) dst[b] = src[b];
}

// --------------------------------------------------------------------------------------------------
// C-ABI

static inline unsigned blocks_for(int64_t n, int per) { return (unsigned)((n + per - 1) / per); }

extern "C" {

int ccx_abi_version(void) { return CCX_ABI_VERSION; }

const char *ccx_strerror(int code)
{
    switch (code) {
    case CCX_OK: return "ok";
    case CCX_ERR_ARG: return "invalid argument";
    case CCX_ERR_CUDA: return "CUDA error (see ccx_last_cuda_error)";
    case CCX_ERR_NOMEM: return "out of device memory";
    case CCX_ERR_STATE: return "invalid handle state";
    case CCX_ERR_UNSUPPORTED: return "unsupported";
    case CCX_ERR_OVERFLOW: return "node pool overflow";
    default: return "unknown error";
    }
}

const char *ccx_last_cuda_error(const ccx_handle *h) { return h ? h->cuda_err : ""; }

int ccx_create(int device_ordinal, ccx_handle **out)
{
    if (!out) return CCX_ERR_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || device_ordinal < 0 || device_ordinal >= count) return e != cudaSuccess ? CCX_ERR_CUDA : CCX_ERR_ARG;
    ccx_handle *h = new (std::nothrow) ccx_handle();
    if (!h) return CCX_ERR_NOMEM;
    h->device = device_ordinal;
    if (cudaSetDevice(device_ordinal) != cudaSuccess) { delete h; return CCX_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device_ordinal) == cudaSuccess) h->num_sms = prop.multiProcessorCount;
    if (cudaMalloc(&h->jump_table, CCX_JT_BYTES) != cudaSuccess) { delete h; return CCX_ERR_NOMEM; }
    k_build_jump_table<<<7, 128>>>(h->jump_table);
    if (cudaMalloc(&h->jump_table3, CCX_JT3_BYTES) != cudaSuccess) { cudaFree(h->jump_table); delete h; return CCX_ERR_NOMEM; }
    k_build_jump_table3<<<28, 128>>>(h->jump_table3);
    if (cudaMalloc(&h->jump_table_wide, CCX_JTW_BYTES) != cudaSuccess) { cudaFree(h->jump_table); cudaFree(h->jump_table3); delete h; return CCX_ERR_NOMEM; }
    k_build_jump_table_wide<<<64, 128>>>((u64 *)h->jump_table_wide, h->jump_table3);
    if (cudaDeviceSynchronize() != cudaSuccess) {
        cudaFree(h->jump_table); cudaFree(h->jump_table3); cudaFree(h->jump_table_wide); delete h; return CCX_ERR_CUDA;
    }
    *out = h;
    return CCX_OK;
}

int ccx_destroy(ccx_handle *h)
{
    if (!h) return CCX_OK;
    cudaSetDevice(h->device);
    ccx_net_free(h);
    ccx_net_tc_free(h);
    ccx_net_acc_free(h);
    ccx_trees_free(h);
    ccx_scratch *s[] = {&h->d_state, &h->d_aux0, &h->d_aux1, &h->d_aux2};
    for (auto *p : s) if (p->ptr) cudaFree(p->ptr);
    if (h->jump_table) cudaFree(h->jump_table);
    if (h->jump_table3) cudaFree(h->jump_table3);
    if (h->jump_table_wide) cudaFree(h->jump_table_wide);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->stream2) cudaStreamDestroy(h->stream2);
    delete h;
    return CCX_OK;
}

int ccx_set_stream(ccx_handle *h, void *cuda_stream)
{
    if (!h) return CCX_ERR_ARG;
    h->stream = (cudaStream_t)cuda_stream;
    return CCX_OK;
}

int ccx_synchronize(ccx_handle *h)
{
    if (!h) return CCX_ERR_ARG;
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

int64_t ccx_launch_count(const ccx_handle *h) { return h ? h->launches : 0; }
int64_t ccx_graph_replays(const ccx_handle *h) { return h ? h->graph_replays : 0; }

int ccx_reset(ccx_handle *h, int64_t n, uint64_t *state, int mode, uint64_t seed, int64_t game_id0)
{
    if (!h || n < 0 || (n && !state) || (mode != CCX_RESET_START && mode != CCX_RESET_RANDOMISED)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_reset<<<blocks_for(n, ENV_THREADS), ENV_THREADS, 0, h->stream>>>((u64 *)state, n, mode, (u32)seed, (u32)(seed >> 32), game_id0);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_movegen(ccx_handle *h, int64_t n, const uint64_t *state, uint64_t *dest_masks)
{
    if (!h || n < 0 || (n && (!state || !dest_masks))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_movegen<<<blocks_for(n, ENV_THREADS), ENV_THREADS, 0, h->stream>>>((const u64 *)state, n, (u64 *)dest_masks, h->jump_table);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_apply(ccx_handle *h, int64_t n, uint64_t *state, const uint8_t *from, const uint8_t *to, uint8_t *winner)
{
    if (!h || n < 0 || (n && (!state || !from || !to || !winner))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_apply<<<blocks_for(n, ENV_THREADS), ENV_THREADS, 0, h->stream>>>((u64 *)state, n, from, to, winner);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_info(ccx_handle *h, int64_t n, const uint64_t *state, int16_t *out)
{
    if (!h || n < 0 || (n && (!state || !out))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_info<<<blocks_for(n, ENV_THREADS), ENV_THREADS, 0, h->stream>>>((const u64 *)state, n, out);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_step_random(ccx_handle *h, int64_t n, uint64_t *state, int64_t game_id0, uint64_t seed, uint32_t step0,
                    int32_t plies, uint64_t *wins, uint64_t *trace, int64_t trace_games)
{
    if (!h || n < 0 || plies < 0 || (n && (!state || !wins)) || (trace_games > 0 && !trace)) return CCX_ERR_ARG;
    if (n == 0 || plies == 0) return CCX_OK;
    // kernel variant (CCX_STEP_VARIANT, for A/B runs; all bit-identical; B200, 65,536 games x 256 plies, profiles/r03d_env_variants.log,
    // variant 11 from profiles/r06_bench_*.json):
    //   11 (default) k_step_random_carry: k_step_random_pick with at most K fill steps per lane and round,      0.427 ms  3.93e10 steps/s
    //                unfinished fills carried into the next round, a shorter per-ply path and fill, the checker
    //                picked speculatively (0.451 ms before); in one wave the wide answer tables (194.5 KB of
    //                dynamic shared memory, 0.528 ms before them).  K = 5 in one
    //                wave, K = 4 beyond (K = 4 / 5 / 6 measured, profiles/r05_carry_k_sweep.log: in one wave 5 beats
    //                4 and 6 by about 1 %; r03d: at 131,072 and 1 M games, two blocks per SM, 4 beats 5 by 1.0 %)
    //   10           k_step_random_pick: one game per lane, pick the checker first, flood-fill only its jumps   0.629 ms  2.67e10
    //   9            k_step_random_wq: all six closures per game from a warp-wide queue of flood fills          2.379 ms  7.05e9
    //                (<PRE> in one wave: 156 KB of shared memory per 448-lane block; beyond, the non-PRE form, two blocks per SM)
    // Every kernel runs one 448-lane block per SM while the batch fits one wave (148 x 448 = 66,304 games), two beyond (MINB = 2:
    // at most 72 registers; k_step_random_carry fits them without spills and gains more there than in one wave).
    const char *ve = getenv("CCX_STEP_VARIANT");
    const int variant = ve ? atoi(ve) : 11;
    if (variant < 9 || variant > 11) return CCX_ERR_ARG;
    const u32 s0 = (u32)seed, s1 = (u32)(seed >> 32);
    const bool tr = trace && trace_games > 0;
    u64 *tp = tr ? (u64 *)trace : nullptr;
    const int64_t tg = tr ? trace_games : 0;
    const bool one_wave = n <= (int64_t)h->num_sms * 448;
    if (variant == 11) {
        if (one_wave && !h->carry_wide_smem) {
            CCX_CUDA(h, cudaFuncSetAttribute(k_step_random_carry<false, 448, 1, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, CCX_WIDE_SMEM_BYTES));
            CCX_CUDA(h, cudaFuncSetAttribute(k_step_random_carry<true, 448, 1, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, CCX_WIDE_SMEM_BYTES));
            h->carry_wide_smem = true;
        }
#define CCX_CARRY_LAUNCH(TR, MINB, K)                                                                                            \
        k_step_random_carry<TR, 448, MINB, K><<<blocks_for(n, 448), 448, (MINB) == 1 ? CCX_WIDE_SMEM_BYTES : 0, h->stream>>>(     \
            (u64 *)state, n, game_id0, s0, s1, step0, plies, (u64 *)wins, tp, tg, h->jump_table3, (const u64 *)h->jump_table_wide)
        if (one_wave) { if (tr) CCX_CARRY_LAUNCH(true, 1, 5); else CCX_CARRY_LAUNCH(false, 1, 5); }
        else { if (tr) CCX_CARRY_LAUNCH(true, 2, 4); else CCX_CARRY_LAUNCH(false, 2, 4); }
#undef CCX_CARRY_LAUNCH
    } else if (variant == 10) {
#define CCX_PICK_LAUNCH(TR, MINB)                                                                                                \
        k_step_random_pick<TR, 448, MINB><<<blocks_for(n, 448), 448, 0, h->stream>>>((u64 *)state, n, game_id0, s0, s1, step0, plies, \
                                                                                     (u64 *)wins, tp, tg, h->jump_table3)
        if (one_wave) { if (tr) CCX_PICK_LAUNCH(true, 1); else CCX_PICK_LAUNCH(false, 1); }
        else { if (tr) CCX_PICK_LAUNCH(true, 2); else CCX_PICK_LAUNCH(false, 2); }
#undef CCX_PICK_LAUNCH
    } else {
#define CCX_WQ_LAUNCH(TR, TPB, MINB, PRE)                                                                                        \
        do {                                                                                                                      \
            static bool attr_set = false;                                                                                         \
            constexpr int DYN = (TPB / 32) * ((PRE) ? 30 : 10) * 32 * 8;                                                           \
            if (!attr_set) {                                                                                                      \
                CCX_CUDA(h, cudaFuncSetAttribute(k_step_random_wq<TR, TPB, MINB, PRE>, cudaFuncAttributeMaxDynamicSharedMemorySize, DYN)); \
                attr_set = true;                                                                                                  \
            }                                                                                                                     \
            k_step_random_wq<TR, TPB, MINB, PRE><<<blocks_for(n, TPB), TPB, DYN, h->stream>>>(                                     \
                (u64 *)state, n, game_id0, s0, s1, step0, plies, (u64 *)wins, tp, tg, h->jump_table3);                              \
        } while (0)
        if (one_wave) { if (tr) CCX_WQ_LAUNCH(true, 448, 1, true); else CCX_WQ_LAUNCH(false, 448, 1, true); }
        else { if (tr) CCX_WQ_LAUNCH(true, 448, 2, false); else CCX_WQ_LAUNCH(false, 448, 2, false); }
#undef CCX_WQ_LAUNCH
    }
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_greedy_candidates(ccx_handle *h, int64_t n, const uint64_t *state, uint64_t *cand_masks)
{
    if (!h || n < 0 || (n && (!state || !cand_masks))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_greedy_candidates<<<blocks_for(n, ENV_THREADS), ENV_THREADS, 0, h->stream>>>((const u64 *)state, n, (u64 *)cand_masks, h->jump_table);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_play_greedy(ccx_handle *h, int64_t n, uint64_t *state, int64_t game_id0, uint64_t seed, int32_t max_plies,
                    uint64_t *counters)
{
    if (!h || n < 0 || max_plies < 0 || (n && !state)) return CCX_ERR_ARG;
    if (n == 0 || max_plies == 0) return CCX_OK;
    // CCX_GREEDY_VARIANT (A/B): 0 = k_play_greedy (byte-table rays, 64-lane blocks); 1 / 2 / 3 = three-layout move generation with
    // 448- / 224- / 128-lane blocks (the 47 KB of tables are per block)
    const char *ve = getenv("CCX_GREEDY_VARIANT");
    const int variant = ve ? atoi(ve) : CCX_GREEDY_DEFAULT_VARIANT;
    if (variant == 1)
        k_play_greedy_tri<448, 2><<<blocks_for(n, 448), 448, 0, h->stream>>>((u64 *)state, n, game_id0, (u32)seed, (u32)(seed >> 32), max_plies, (u64 *)counters, h->jump_table3);
    else if (variant == 2)
        k_play_greedy_tri<224, 4><<<blocks_for(n, 224), 224, 0, h->stream>>>((u64 *)state, n, game_id0, (u32)seed, (u32)(seed >> 32), max_plies, (u64 *)counters, h->jump_table3);
    else if (variant == 3)
        k_play_greedy_tri<128, 4><<<blocks_for(n, 128), 128, 0, h->stream>>>((u64 *)state, n, game_id0, (u32)seed, (u32)(seed >> 32), max_plies, (u64 *)counters, h->jump_table3);
    else
        k_play_greedy<<<blocks_for(n, ENV_THREADS), ENV_THREADS, 0, h->stream>>>((u64 *)state, n, game_id0, (u32)seed,
                                                                                  (u32)(seed >> 32), max_plies, (u64 *)counters, h->jump_table);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_encode(ccx_handle *h, int64_t n, const uint64_t *state, void *out, int dtype)
{
    if (!h || n < 0 || (n && (!state || !out))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    constexpr int SMEM = 128 * 343;      // 43,904 B for every dtype (G = 128 / 64 / 32)
    switch (dtype) {
    case CCX_DTYPE_U8:
        k_encode<uint8_t, 128><<<blocks_for(n, 128), ENC_THREADS, SMEM, h->stream>>>((const u64 *)state, n, (uint8_t *)out);
        break;
    case CCX_DTYPE_BF16:
        k_encode<__nv_bfloat16, 64><<<blocks_for(n, 64), ENC_THREADS, SMEM, h->stream>>>((const u64 *)state, n, (__nv_bfloat16 *)out);
        break;
    case CCX_DTYPE_F32:
        k_encode<float, 32><<<blocks_for(n, 32), ENC_THREADS, SMEM, h->stream>>>((const u64 *)state, n, (float *)out);
        break;
    default:
        return CCX_ERR_ARG;
    }
    CCX_LAUNCHED(h);
    return CCX_OK;
}

// ---- host-buffer variants ---------------------------------------------------------------------------

int ccx_movegen_host(ccx_handle *h, int64_t n, const uint64_t *state_host, uint64_t *dest_masks_host)
{
    if (!h || n < 0 || (n && (!state_host || !dest_masks_host))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    size_t sb = (size_t)n * CCX_STATE_WORDS * 8, mb = (size_t)n * 6 * 8;
    int rc;
    if ((rc = ccx_reserve(h, h->d_state, sb)) || (rc = ccx_reserve(h, h->d_aux0, mb))) return rc;
    // only words 0-4 are read by movegen
    CCX_CUDA(h, cudaMemcpyAsync(h->d_state.ptr, state_host, (size_t)n * 5 * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ccx_movegen(h, n, (const uint64_t *)h->d_state.ptr, (uint64_t *)h->d_aux0.ptr))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(dest_masks_host, h->d_aux0.ptr, mb, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

int ccx_apply_host(ccx_handle *h, int64_t n, uint64_t *state_host, const uint8_t *from_host, const uint8_t *to_host,
                   uint8_t *winner_host)
{
    if (!h || n < 0 || (n && (!state_host || !from_host || !to_host || !winner_host))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    size_t sb = (size_t)n * CCX_STATE_WORDS * 8;
    int rc;
    if ((rc = ccx_reserve(h, h->d_state, sb)) || (rc = ccx_reserve(h, h->d_aux0, (size_t)n)) ||
        (rc = ccx_reserve(h, h->d_aux1, (size_t)n)) || (rc = ccx_reserve(h, h->d_aux2, (size_t)n))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(h->d_state.ptr, state_host, sb, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaMemcpyAsync(h->d_aux0.ptr, from_host, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaMemcpyAsync(h->d_aux1.ptr, to_host, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ccx_apply(h, n, (uint64_t *)h->d_state.ptr, (const uint8_t *)h->d_aux0.ptr, (const uint8_t *)h->d_aux1.ptr,
                        (uint8_t *)h->d_aux2.ptr))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(state_host, h->d_state.ptr, sb, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaMemcpyAsync(winner_host, h->d_aux2.ptr, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

int ccx_step_random_host(ccx_handle *h, int64_t n, uint64_t *state_host, int64_t game_id0, uint64_t seed, uint32_t step0,
                         int32_t plies, uint64_t *wins_host)
{
    if (!h || n < 0 || plies < 0 || (n && (!state_host || !wins_host))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    size_t sb = (size_t)n * CCX_STATE_WORDS * 8, hot = (size_t)n * 5 * 8;
    int rc;
    if ((rc = ccx_reserve(h, h->d_state, sb)) || (rc = ccx_reserve(h, h->d_aux0, 16))) return rc;
    // the step touches words 0-4 only: 40 B per game each way
    CCX_CUDA(h, cudaMemcpyAsync(h->d_state.ptr, state_host, hot, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaMemcpyAsync(h->d_aux0.ptr, wins_host, 16, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ccx_step_random(h, n, (uint64_t *)h->d_state.ptr, game_id0, seed, step0, plies, (uint64_t *)h->d_aux0.ptr,
                              nullptr, 0))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(state_host, h->d_state.ptr, hot, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaMemcpyAsync(wins_host, h->d_aux0.ptr, 16, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

int ccx_greedy_candidates_host(ccx_handle *h, int64_t n, const uint64_t *state_host, uint64_t *cand_masks_host)
{
    if (!h || n < 0 || (n && (!state_host || !cand_masks_host))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    size_t sb = (size_t)n * CCX_STATE_WORDS * 8, mb = (size_t)n * 6 * 8;
    int rc;
    if ((rc = ccx_reserve(h, h->d_state, sb)) || (rc = ccx_reserve(h, h->d_aux0, mb))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(h->d_state.ptr, state_host, (size_t)n * 5 * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ccx_greedy_candidates(h, n, (const uint64_t *)h->d_state.ptr, (uint64_t *)h->d_aux0.ptr))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(cand_masks_host, h->d_aux0.ptr, mb, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

int ccx_info_host(ccx_handle *h, int64_t n, const uint64_t *state_host, int16_t *out_host)
{
    if (!h || n < 0 || (n && (!state_host || !out_host))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    size_t sb = (size_t)n * CCX_STATE_WORDS * 8, ob = (size_t)n * 5 * sizeof(int16_t);
    int rc;
    if ((rc = ccx_reserve(h, h->d_state, sb)) || (rc = ccx_reserve(h, h->d_aux0, ob))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(h->d_state.ptr, state_host, (size_t)n * 5 * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ccx_info(h, n, (const uint64_t *)h->d_state.ptr, (int16_t *)h->d_aux0.ptr))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(out_host, h->d_aux0.ptr, ob, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

int ccx_encode_host(ccx_handle *h, int64_t n, const uint64_t *state_host, void *out_host, int dtype)
{
    if (!h || n < 0 || (n && (!state_host || !out_host))) return CCX_ERR_ARG;
    if (dtype < CCX_DTYPE_U8 || dtype > CCX_DTYPE_F32) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    size_t esz = dtype == CCX_DTYPE_U8 ? 1 : dtype == CCX_DTYPE_BF16 ? 2 : 4;
    size_t sb = (size_t)n * CCX_STATE_WORDS * 8, ob = (size_t)n * 343 * esz;
    int rc;
    if ((rc = ccx_reserve(h, h->d_state, sb)) || (rc = ccx_reserve(h, h->d_aux0, ob))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(h->d_state.ptr, state_host, (size_t)n * 5 * 8, cudaMemcpyHostToDevice, h->stream));
    if ((rc = ccx_encode(h, n, (const uint64_t *)h->d_state.ptr, h->d_aux0.ptr, dtype))) return rc;
    CCX_CUDA(h, cudaMemcpyAsync(out_host, h->d_aux0.ptr, ob, cudaMemcpyDeviceToHost, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    return CCX_OK;
}

}  // extern "C"

// weak defaults so that libccx.so links before the MCTS / net translation units exist
__attribute__((weak)) void ccx_net_free(ccx_handle *) {}
__attribute__((weak)) void ccx_trees_free(ccx_handle *) {}
__attribute__((weak)) void ccx_trees_set_uids(ccx_handle *, const int64_t *) {}
__attribute__((weak)) void ccx_net_tc_free(ccx_handle *) {}
