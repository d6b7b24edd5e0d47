// ccx_selfplay.cu — batched selfplay.selfplay() bookkeeping (selfplay.py:11-133) and the trajectory
// packer feeding utils.convert_to_train_data's format (utils.py:60-73).
//
// One game slot per tree.  Per ply-iteration the host enqueues: MCTS over all slots that are past the
// random opening (ccx_mcts_begin with min_ply = INITIAL_RANDOM_MOVES) -> ccx_selfplay_advance (random
// opening move or a move sampled from pi, record (state, visits), repetition / progress / win rules)
// -> ccx_selfplay_finish (label the finished game's records with the outcome, or drop them for a
// discarded game, and restart the slot).  Nothing on this path touches the host.
#include "ccx_device.cuh"
#include "ccx_internal.h"
#include <math_constants.h>

#define FULL 0xFFFFFFFFu
#define SP_WARPS 4

// record flags
enum { REC_NONE = 0, REC_PENDING = 1, REC_WIN = 2, REC_LOSS = 3, REC_DROPPED = 4, REC_TAU_DET = 0x10 };

__device__ __forceinline__ double u01(u32 x) { return (double)x / 4294967296.0; }

// ---- Dirichlet noise: raw Gamma(alpha, 1) draws, normalised later over the root's edge count -------------
// Marsaglia-Tsang (2000) for alpha + 1 with the U^(1/alpha) boost for alpha < 1; Philox counter RNG.
__global__ void __launch_bounds__(128)
k_gamma_noise(double *__restrict__ out, int64_t n, int stride, double alpha, u32 k0, u32 k1, u32 iter, int64_t uid0,
              const int64_t *__restrict__ slot_ids)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * stride) return;
    int64_t tree = t / stride; int j = (int)(t % stride);
    u64 uid = (u64)(slot_ids ? slot_ids[tree] : uid0 + tree);
    const double d = alpha + 1.0 - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    double g = 0.0;
    for (u32 attempt = 0; attempt < 64; attempt++) {
        Philox4 r = philox4x32_10(k0, k1, iter, 0x100u + (u32)j * 64u + attempt, (u32)uid, (u32)(uid >> 32) ^ 0xD1A1u);
        double u1 = (u01(r.x) + 1.0 / 8589934592.0), u2 = u01(r.y);
        double x = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);                 // Box-Muller
        double v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        double u = u01(r.z) + 1.0 / 8589934592.0;
        if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) {
            double ub = u01(r.w) + 1.0 / 8589934592.0;
            g = d * v * pow(ub, 1.0 / alpha);
            break;
        }
    }
    out[t] = g;
}

// np.random.choice(294, p=pi) with pi = N^(1/tau) / sum (MCTS.py:131-140), warp-cooperative: each lane owns ten
// consecutive actions, an inclusive scan of the lane sums locates the lane whose interval holds rnd * total.
__device__ __forceinline__ int sample_action(const u32 *__restrict__ vis, bool det, double inv_tau, u32 rnd, int lane)
{
    double w[10], local = 0.0;
#pragma unroll
    for (int q = 0; q < 10; q++) {
        int a = lane * 10 + q;
        double N = a < CCX_NUM_ACTIONS ? (double)vis[a] : 0.0;
        w[q] = det ? pow(N, inv_tau) : N;
        local += w[q];
    }
    double incl = local;                                  // inclusive warp scan of the lane sums
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { double o = __shfl_up_sync(FULL, incl, off); if (lane >= off) incl += o; }
    double total = __shfl_sync(FULL, incl, 31);
    double target = u01(rnd) * total;                     // np.random.choice(294, p=pi) (MCTS.py:140)
    double excl = incl - local;
    int mine = -1;
    if (target >= excl && target < incl) {
        double acc = excl;
#pragma unroll
        for (int q = 0; q < 10; q++) { acc += w[q]; if (mine < 0 && w[q] > 0.0 && target < acc) mine = lane * 10 + q; }
    }
    // lowest lane that found an action wins; fall back to the most visited action on rounding edge cases
    u32 have = __ballot_sync(FULL, mine >= 0);
    if (have) return __shfl_sync(FULL, mine, __ffs(have) - 1);
    u32 bestN = 0; int besta = 0;
#pragma unroll
    for (int q = 0; q < 10; q++) { int a = lane * 10 + q; if (a < CCX_NUM_ACTIONS && vis[a] > bestN) { bestN = vis[a]; besta = a; } }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        u32 oN = __shfl_xor_sync(FULL, bestN, off); int oa = __shfl_xor_sync(FULL, besta, off);
        if (oN > bestN || (oN == bestN && oa < besta)) { bestN = oN; besta = oa; }
    }
    return besta;
}

// ---- advance one ply per running game -----------------------------------------------------------------------
// warp per game; visits = MCTS result of this iteration (ignored for opening plies).
__global__ void __launch_bounds__(32 * SP_WARPS)
k_selfplay_advance(u64 *__restrict__ st, int64_t n, const u32 *__restrict__ visits, const int32_t *__restrict__ tree_nodes,
                   u32 k0, u32 k1, int iter, int64_t uid0, const int64_t *__restrict__ serial, int64_t total_slots,
                   int random_plies, int tau_switch, int move_limit,
                   u64 *__restrict__ rec_state, uint16_t *__restrict__ rec_visits, uint8_t *__restrict__ rec_flag,
                   int rec_iters, u64 *__restrict__ counters, u32 *__restrict__ move_log, const uint8_t *__restrict__ jt,
                   const int64_t *__restrict__ slot_ids)
{
    __shared__ __align__(16) uint8_t sT[CCX_JT_BYTES];
    for (int q = threadIdx.x; q < CCX_JT_BYTES / 16; q += blockDim.x) reinterpret_cast<uint4 *>(sT)[q] = reinterpret_cast<const uint4 *>(jt)[q];
    __syncthreads();
    int64_t g = (int64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (g >= n) return;
    u64 meta = st[4 * n + g];
    if ((meta >> 56) != CCX_ST_RUNNING) return;
    bool p2 = (meta >> 48) & 1;
    u64 occ1 = st[0 * n + g], occ2 = st[1 * n + g], c1 = st[2 * n + g], c2 = st[3 * n + g];
    Game gm;
    gm.meta = meta;
    gm.occ_me = p2 ? occ2 : occ1; gm.occ_op = p2 ? occ1 : occ2;
    gm.cells_me = p2 ? c2 : c1;   gm.cells_op = p2 ? c1 : c2;
    u64 lo = st[5 * n + g], hi = st[6 * n + g], aux = st[7 * n + g];
    int ply = (int)((meta >> 32) & 0xFFFF);
    u64 uid = (u64)(serial[g] * total_slots + (slot_ids ? slot_ids[g] : uid0 + g));      // unique per game instance
    int id, from, to;
    int recorded = (int)((aux >> 32) & 0xFFFF);
    if (ply < random_plies) {
        // selfplay.make_random_move (selfplay.py:83-104)
        u64 dest[6];
        movegen_rays(gm.occ_me | gm.occ_op, gm.cells_me, dest, sT);
        u32 nonempty = 0;
#pragma unroll
        for (int k = 0; k < 6; k++) nonempty += dest[k] != 0;
        Philox4 r = philox4x32_10(k0, k1, (u32)ply, 0u, (u32)uid, (u32)(uid >> 32));
        id = pick_random(gm, dest, nonempty, r.x, r.y, from, to);
    } else {
        if (tree_nodes[g] < 0) {         // pool overflow: the search result is unusable -> discard the game (counted by k_selfplay_finish)
            if (lane == 0) st[4 * n + g] = (meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)CCX_ST_OVERFLOW << 56);
            return;
        }
        // pi = N^(1/tau) / sum (MCTS.py:131-137); tau = DET_TREE_TAU once len(play_history) + 6 > 16 (selfplay.py:62-65)
        bool det = recorded + random_plies > tau_switch;
        double inv_tau = det ? 1.0 / 0.01 : 1.0;
        const u32 *vis = visits + g * CCX_NUM_ACTIONS;
        Philox4 r = philox4x32_10(k0, k1, (u32)ply, 3u, (u32)uid, (u32)(uid >> 32));
        int action = sample_action(vis, det, inv_tau, r.x, lane);
        id = action / 49;                                     // utils.decode_checker_index (utils.py:175-183)
        int off = action % 49;
        to = (off / 7) * 8 + (off % 7);
        from = (int)((gm.cells_me >> (8 * id)) & 0xFF);
        // play_history.append((root.state, pi))  (selfplay.py:128)
        {
            int64_t rec = (int64_t)(iter % rec_iters) * n + g;          // ring over iterations
            if (lane < 5) rec_state[rec * 5 + lane] = st[lane * n + g];
            for (int a = lane; a < CCX_NUM_ACTIONS; a += 32) rec_visits[rec * CCX_NUM_ACTIONS + a] = (uint16_t)vis[a];
            if (lane == 0) rec_flag[rec] = (uint8_t)(REC_PENDING | (det ? REC_TAU_DET : 0));
        }
        recorded++;
    }
    __syncwarp();
    if (lane != 0) return;
    int mover = p2 ? 1 : 0;
    apply_move(gm, id, from, to);
    push_hist(lo, hi, to);
    ply++;
    int status = CCX_ST_RUNNING;
    // repetition rule (selfplay.py:40-47): fires from 15 stored plies on
    if (ply >= 15 && repetition_stop(lo, hi)) status = CCX_ST_REPETITION;
    u32 useless = (u32)(aux & 0xFFFF);
    u32 prog[2] = {(u32)((aux >> 16) & 0xFF), (u32)((aux >> 24) & 0xFF)};
    if (status == CCX_ST_RUNNING) {
        // progress bookkeeping (selfplay.py:50-55); after apply_move the mover's pieces are occ_op
        u32 p = (u32)__popcll(gm.occ_op & (mover ? CCX_TARGET_P2 : CCX_TARGET_P1));
        if (p > prog[mover]) { useless = useless * 5u / 6u; prog[mover] = p; }
        else useless++;
        int win = winner_of(gm);                                         // selfplay.py:67-69
        if (win) status = win;
        else if ((int)useless >= move_limit) status = CCX_ST_MOVE_LIMIT;  // selfplay.py:72-74
    }
    aux = (u64)(useless & 0xFFFF) | ((u64)prog[0] << 16) | ((u64)prog[1] << 24) | ((u64)(recorded & 0xFFFF) << 32);
    gm.meta = (gm.meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)status << 56);
    bool np2 = (gm.meta >> 48) & 1;
    st[0 * n + g] = np2 ? gm.occ_op : gm.occ_me; st[1 * n + g] = np2 ? gm.occ_me : gm.occ_op;
    st[2 * n + g] = np2 ? gm.cells_op : gm.cells_me; st[3 * n + g] = np2 ? gm.cells_me : gm.cells_op;
    st[4 * n + g] = gm.meta; st[5 * n + g] = lo; st[6 * n + g] = hi; st[7 * n + g] = aux;
    atomicAdd(&counters[0], 1ULL);                                       // plies played
    if (move_log)       // from | to<<8 | status after the move<<16 | 1<<24 (valid) | recorded-by-MCTS<<25
        move_log[(int64_t)(iter % rec_iters) * n + g] = (u32)from | ((u32)to << 8) | ((u32)status << 16) | (1u << 24) |
                                          ((ply - 1 >= random_plies ? 1u : 0u) << 25);
}

// ---- Game.start (game.py:58-100) for arena / evaluation games: one ply per running game ------------------------
// visits != NULL: the mover is an AiPlayer (player.py:136-166): MCTS.search was run on the unexpanded root, the move is
// sampled from pi = N^(1/tau), tau = DET_TREE_TAU once total_moves > TOTAL_MOVES_TILL_TAU0 (player.py:151-154).
// visits == NULL: the mover is the GreedyPlayer (player.py:72-76, 99-121): uniform pick among filtered_best_moves.
// Then game.py:65-89: winner, 16-deque of destinations + repetition stop, optional move limit.
// counters: [0] plies, [1] P1 wins, [2] P2 wins, [3] stopped (repetition / move limit / overflow / no moves)
__global__ void __launch_bounds__(32 * SP_WARPS)
k_game_advance(u64 *__restrict__ st, int64_t n, const u32 *__restrict__ visits, const int32_t *__restrict__ tree_nodes,
               u32 k0, u32 k1, int64_t uid0, double tau, int tau0_after, int move_limit, u64 *__restrict__ counters,
               const uint8_t *__restrict__ jt)
{
    __shared__ __align__(16) uint8_t sT[CCX_JT_BYTES];
    for (int q = threadIdx.x; q < CCX_JT_BYTES / 16; q += blockDim.x) reinterpret_cast<uint4 *>(sT)[q] = reinterpret_cast<const uint4 *>(jt)[q];
    __syncthreads();
    int64_t g = (int64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (g >= n) return;
    u64 meta = st[4 * n + g];
    if ((meta >> 56) != CCX_ST_RUNNING) return;
    bool p2 = (meta >> 48) & 1;
    u64 occ1 = st[0 * n + g], occ2 = st[1 * n + g], c1 = st[2 * n + g], c2 = st[3 * n + g];
    Game gm;
    gm.meta = meta;
    gm.occ_me = p2 ? occ2 : occ1; gm.occ_op = p2 ? occ1 : occ2;
    gm.cells_me = p2 ? c2 : c1;   gm.cells_op = p2 ? c1 : c2;
    u64 lo = st[5 * n + g], hi = st[6 * n + g];
    int ply = (int)((meta >> 32) & 0xFFFF);
    u64 uid = (u64)(uid0 + g);
    int id, from, to, status = CCX_ST_RUNNING;
    if (visits) {
        if (tree_nodes && tree_nodes[g] < 0) status = CCX_ST_OVERFLOW;          // pool overflow: the search result is unusable
        else {
            bool det = tau != 1.0 || ply > tau0_after;                          // total_moves == plies played so far
            double inv_tau = ply > tau0_after ? 1.0 / 0.01 : 1.0 / tau;
            Philox4 r = philox4x32_10(k0, k1, (u32)ply, 4u, (u32)uid, (u32)(uid >> 32));
            int action = sample_action(visits + g * CCX_NUM_ACTIONS, det, inv_tau, r.x, lane);
            id = action / 49;
            int off = action % 49;
            to = (off / 7) * 8 + (off % 7);
            from = (int)((gm.cells_me >> (8 * id)) & 0xFF);
        }
    } else {
        u64 dest[6], cand[6];
        movegen_rays(gm.occ_me | gm.occ_op, gm.cells_me, dest, sT);
        int total = greedy_candidates(gm, dest, cand);
        if (total == 0) status = CCX_ST_NO_MOVES;                               // the reference raises (player.py:113)
        else {
            Philox4 r = philox4x32_10(k0, k1, (u32)ply, 1u, (u32)uid, (u32)(uid >> 32));
            id = pick_candidate(gm, cand, total, r.x, from, to);                // player.py:121
        }
    }
    __syncwarp();
    if (lane != 0) return;
    if (status == CCX_ST_RUNNING) {
        apply_move(gm, id, from, to);                                           // game.py:65
        push_hist(lo, hi, to);
        ply++;
        int win = winner_of(gm);
        if (win) status = win;                                                  // game.py:70-71
        else if (ply >= 16 && repetition_stop(lo, hi)) status = CCX_ST_REPETITION;       // game.py:73-82
        else if (move_limit > 0 && ply >= move_limit) status = CCX_ST_MOVE_LIMIT;        // game.py:84-89
        atomicAdd(&counters[0], 1ULL);
    }
    if (status == CCX_ST_WON_P1) atomicAdd(&counters[1], 1ULL);
    else if (status == CCX_ST_WON_P2) atomicAdd(&counters[2], 1ULL);
    else if (status != CCX_ST_RUNNING) atomicAdd(&counters[3], 1ULL);
    gm.meta = (gm.meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)status << 56);
    bool np2 = (gm.meta >> 48) & 1;
    st[0 * n + g] = np2 ? gm.occ_op : gm.occ_me; st[1 * n + g] = np2 ? gm.occ_me : gm.occ_op;
    st[2 * n + g] = np2 ? gm.cells_op : gm.cells_me; st[3 * n + g] = np2 ? gm.cells_me : gm.cells_op;
    st[4 * n + g] = gm.meta; st[5 * n + g] = lo; st[6 * n + g] = hi;
}

// ---- finish: label or drop the records of every game that ended this iteration, restart the slot -----------
// counters: [0] plies, [1] P1 wins, [2] P2 wins, [3] discarded by repetition, [4] discarded by the progress
// limit, [5] discarded by pool overflow, [6] records kept, [7] games finished (kept)
__global__ void __launch_bounds__(128)
k_selfplay_finish(u64 *__restrict__ st, int64_t n, int iter, int32_t *__restrict__ start_iter, int64_t *__restrict__ serial,
                  const u64 *__restrict__ rec_state, uint8_t *__restrict__ rec_flag, int rec_iters, int max_game_iters, int restart,
                  long long *__restrict__ starts_left, u64 *__restrict__ counters)
{
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    u64 meta = st[4 * n + g];
    int status = (int)(meta >> 56);
    const int first = start_iter[g];
    if (status == CCX_ST_RUNNING) {
        // a game about to outgrow the record ring is discarded while all of its records are still intact
        if (max_game_iters <= 0 || iter - first + 1 < max_game_iters) return;
        status = CCX_ST_OVERFLOW;
        st[4 * n + g] = (meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)CCX_ST_OVERFLOW << 56);
    }
    if (first > iter) return;                                     // ended earlier and was not allowed to restart: already accounted for
    // a resignation (ccx_selfplay_resign) is the other player's win for the labels and the counters
    if (status == CCX_ST_RESIGN_WON_P1) status = CCX_ST_WON_P1;
    else if (status == CCX_ST_RESIGN_WON_P2) status = CCX_ST_WON_P2;
    int kept = 0;
    for (int it = (iter - first >= rec_iters) ? iter - rec_iters + 1 : first; it <= iter; it++) {
        int64_t rec = (int64_t)(it % rec_iters) * n + g;
        uint8_t f = rec_flag[rec];
        if ((f & 0xF) != REC_PENDING) continue;
        if (status == CCX_ST_WON_P1 || status == CCX_ST_WON_P2) {
            // reward from the point of view of the side to move in the recorded position
            // (utils.convert_to_train_data, utils.py:65-71, with utils.get_p1_winloss_reward, utils.py:34-44)
            int mover = (int)((rec_state[rec * 5 + 4] >> 48) & 1) + 1;
            rec_flag[rec] = (uint8_t)((f & 0xF0) | (mover == status ? REC_WIN : REC_LOSS));
            kept++;
        } else {
            rec_flag[rec] = (uint8_t)((f & 0xF0) | REC_DROPPED);       // `return None, None` (selfplay.py:47,74)
        }
    }
    if (status == CCX_ST_WON_P1) atomicAdd(&counters[1], 1ULL);
    else if (status == CCX_ST_WON_P2) atomicAdd(&counters[2], 1ULL);
    else if (status == CCX_ST_REPETITION) atomicAdd(&counters[3], 1ULL);
    else if (status == CCX_ST_MOVE_LIMIT) atomicAdd(&counters[4], 1ULL);
    else if (status == CCX_ST_OVERFLOW) atomicAdd(&counters[5], 1ULL);
    if (kept) { atomicAdd(&counters[6], (u64)kept); atomicAdd(&counters[7], 1ULL); }
    // train.py:58-64 plays exactly num_self_play games: with a budget of starts, WHICH of this iteration's ended slots restart is
    // decided by k_selfplay_restart in slot order (deterministic; an atomic ticket here would make it a race)
    if (restart && starts_left) { start_iter[g] = 0x7FFFFFFE; return; }
    const bool again = restart != 0;
    start_iter[g] = again ? iter + 1 : 0x7FFFFFFF;               // records settled; a slot that stays ended is never accounted twice
    if (again) {
        st[0 * n + g] = CCX_START_OCC1; st[1 * n + g] = CCX_START_OCC2;
        st[2 * n + g] = CCX_START_CELLS1; st[3 * n + g] = CCX_START_CELLS2;
        st[4 * n + g] = CCX_START_META; st[5 * n + g] = CCX_HIST_EMPTY; st[6 * n + g] = CCX_HIST_EMPTY; st[7 * n + g] = 0;
        serial[g] += 1;
    }
}

// Restarts under a budget: the slots that ended in this iteration (start_iter == 0x7FFFFFFE) restart in slot order while
// *starts_left > 0; the rest stay ended.  One block scans all slots (n is a few thousand).
__global__ void __launch_bounds__(1024)
k_selfplay_restart(u64 *__restrict__ st, int64_t n, int iter, int32_t *__restrict__ start_iter, int64_t *__restrict__ serial,
                   long long *__restrict__ starts_left)
{
    __shared__ int warp_tot[32];
    __shared__ long long budget_s;
    __shared__ int base_s;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) { budget_s = *starts_left; base_s = 0; }
    __syncthreads();
    const long long budget = budget_s > 0 ? budget_s : 0;
    for (int64_t g0 = 0; g0 < n; g0 += 1024) {
        const int64_t g = g0 + t;
        const bool cand = g < n && start_iter[g] == 0x7FFFFFFE;
        const unsigned b = __ballot_sync(0xFFFFFFFFu, cand);
        if (lane == 0) warp_tot[warp] = __popc(b);
        __syncthreads();
        int before = base_s;
        for (int w = 0; w < warp; w++) before += warp_tot[w];
        const int rank = before + __popc(b & ((1u << lane) - 1u));
        if (cand) {
            if ((long long)rank < budget) {
                st[0 * n + g] = CCX_START_OCC1; st[1 * n + g] = CCX_START_OCC2;
                st[2 * n + g] = CCX_START_CELLS1; st[3 * n + g] = CCX_START_CELLS2;
                st[4 * n + g] = CCX_START_META; st[5 * n + g] = CCX_HIST_EMPTY; st[6 * n + g] = CCX_HIST_EMPTY; st[7 * n + g] = 0;
                start_iter[g] = iter + 1;
                serial[g] += 1;
            } else {
                start_iter[g] = 0x7FFFFFFF;
            }
        }
        __syncthreads();
        if (t == 0) { int tot = 0; for (int w = 0; w < 32; w++) tot += warp_tot[w]; base_s += tot; }
        __syncthreads();
    }
    if (t == 0) *starts_left = budget_s - (long long)(base_s < budget ? base_s : budget);
}

// ---- opt-in resignation (include/ccx.h, "self-play resignation") ---------------------------------------------------------------
// resign_state row (int64[CCX_RESIGN_WORDS]): [0] serial of the game it belongs to (-1 = none); [1] flags: bit 0 probe, bits 1-2
// would-be resigner (0 none, 1 player 1, 2 player 2), bits 8 + 8p streak of player p, bits 24 + 4p ring position, bits 32 + 4p
// values in the ring (<= plies); [2 + p] window minimum of player p (float64 bits); [4 + 8p .. 11 + 8p] player p's last r values.
enum { RS_SERIAL = 0, RS_FLAGS = 1, RS_WMIN = 2, RS_RING = 4 };
#define RS_PURPOSE 0x52534750u

__device__ __forceinline__ void resign_slot_init(int64_t *__restrict__ row, int64_t serial, u32 k0, u32 k1, u64 sid, double probe)
{
    const Philox4 r = philox4x32_10(k0, k1, (u32)sid, (u32)(sid >> 32), (u32)serial, RS_PURPOSE);
    row[RS_SERIAL] = serial;
    row[RS_FLAGS] = u01(r.x) < probe ? 1 : 0;
    row[RS_WMIN] = row[RS_WMIN + 1] = __double_as_longlong(CUDART_INF);
}

// ---- opt-in playout cap randomization (include/ccx.h, "self-play playout cap randomization") ------------------------------------
#define PC_PURPOSE 0x50430000u      // + ply: disjoint from RS_PURPOSE for every 16-bit ply count

// one thread per slot: the slot's budget for this iteration's search; the searching slots add to {full, fast} (one atomic per warp)
__global__ void __launch_bounds__(128)
k_selfplay_playout_cap(const u64 *__restrict__ st, int64_t n, u32 k0, u32 k1, int64_t uid0, const int64_t *__restrict__ slot_ids,
                       const int64_t *__restrict__ serial, int min_ply, double p, int full_budget, int fast_budget,
                       int32_t *__restrict__ budget, u64 *__restrict__ counters, uint8_t *__restrict__ keep)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    u32 full = 0, fast = 0;
    if (g < n) {
        const u64 meta = st[4 * n + g];
        const int ply = (int)((meta >> 32) & 0xFFFF);
        const u64 sid = (u64)(slot_ids ? slot_ids[g] : uid0 + g);
        const Philox4 r = philox4x32_10(k0, k1, (u32)sid, (u32)(sid >> 32), (u32)serial[g], PC_PURPOSE + (u32)ply);
        const bool is_full = u01(r.x) < p;
        const bool searches = (meta >> 56) == CCX_ST_RUNNING && ply >= min_ply;
        budget[g] = is_full || !searches ? full_budget : fast_budget;
        if (keep) keep[g] = is_full || !searches;
        full = searches && is_full;
        fast = searches && !is_full;
    }
    full = __reduce_add_sync(FULL, full);
    fast = __reduce_add_sync(FULL, fast);
    if ((threadIdx.x & 31) == 0) {
        if (full) atomicAdd(&counters[0], (u64)full);
        if (fast) atomicAdd(&counters[1], (u64)fast);
    }
}

// warp per slot: r of the slot's tree (the sums in the order include/ccx.h fixes), then lane 0 updates the mover's streak and window
__global__ void __launch_bounds__(32 * SP_WARPS)
k_selfplay_resign(ccx_root_view tv, u64 *__restrict__ st, int64_t n, u32 k0, u32 k1, int64_t uid0, const int64_t *__restrict__ slot_ids,
                  const int64_t *__restrict__ serial, double threshold, int plies, double probe, int64_t *__restrict__ rs,
                  double *__restrict__ value_out, u64 *__restrict__ counters)
{
    const int64_t g = (int64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= n) return;
    int64_t *row = rs + g * CCX_RESIGN_WORDS;
    if (lane == 0 && row[RS_SERIAL] != serial[g])
        resign_slot_init(row, serial[g], k0, k1, (u64)(slot_ids ? slot_ids[g] : uid0 + g), probe);
    const u64 meta = st[4 * n + g];
    bool has = (meta >> 56) == CCX_ST_RUNNING && tv.meta[g * 8 + 2] == 0;
    double r = CUDART_NAN;
    if (has) {
        const u64 info = tv.node[g * (int64_t)tv.npt * 6 + 5];
        const int ne = (int)((info >> 32) & 0xFF), eb = (int)(u32)info;
        const u32 *eN = tv.eN + g * (int64_t)tv.ept + eb;
        const double *eW = tv.eW + g * (int64_t)tv.ept + eb;
        double snq = 0.0, sn = 0.0;
        u32 bestN = 0; int bestj = 0x7FFFFFFF; double bestq = 0.0;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int j = lane + 32 * c;
            const u32 N = j < ne ? eN[j] : 0u;
            const double q = N ? __ddiv_rn(eW[j], (double)N) : 0.0;        // ccx_mcts_finalize's Q
            snq = __dadd_rn(snq, __dmul_rn((double)N, q));
            sn = __dadd_rn(sn, (double)N);
            if (j < ne && (bestj == 0x7FFFFFFF || N > bestN)) { bestN = N; bestj = j; bestq = q; }
        }
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            snq = __dadd_rn(snq, __shfl_xor_sync(FULL, snq, off));
            sn = __dadd_rn(sn, __shfl_xor_sync(FULL, sn, off));
            const u32 oN = __shfl_xor_sync(FULL, bestN, off);
            const int oj = __shfl_xor_sync(FULL, bestj, off);
            const double oq = __shfl_xor_sync(FULL, bestq, off);
            if (oj != 0x7FFFFFFF && (bestj == 0x7FFFFFFF || oN > bestN || (oN == bestN && oj < bestj))) { bestN = oN; bestj = oj; bestq = oq; }
        }
        has = sn > 0.0;
        if (has) r = fmax(__ddiv_rn(snq, sn), bestq);
    }
    if (lane != 0) return;
    if (value_out) value_out[g] = r;
    if (!has) return;
    const int p = (int)((meta >> 48) & 1);
    u64 f = (u64)row[RS_FLAGS];
    int pos = (int)((f >> (24 + 4 * p)) & 0xF), filled = (int)((f >> (32 + 4 * p)) & 0xF), streak = (int)((f >> (8 + 8 * p)) & 0xFF);
    double *ring = reinterpret_cast<double *>(row + RS_RING + 8 * p);
    ring[pos] = r;
    pos = pos + 1 == plies ? 0 : pos + 1;
    if (filled < plies) filled++;
    if (filled == plies) {
        double wmax = ring[0];
        for (int k = 1; k < plies; k++) wmax = fmax(wmax, ring[k]);
        double *wmin = reinterpret_cast<double *>(row + RS_WMIN + p);
        *wmin = fmin(*wmin, wmax);
    }
    streak = r < threshold ? min(streak + 1, plies) : 0;
    if (streak >= plies) {
        if (f & 1) {
            if (((f >> 1) & 3) == 0) f |= (u64)(p + 1) << 1;            // a probe only remembers who would have resigned
        } else {
            st[4 * n + g] = (meta & 0x00FFFFFFFFFFFFFFULL) | ((u64)(p ? CCX_ST_RESIGN_WON_P1 : CCX_ST_RESIGN_WON_P2) << 56);
            atomicAdd(&counters[0], 1ULL);
        }
    }
    f &= ~((0xFFULL << (8 + 8 * p)) | (0xFULL << (24 + 4 * p)) | (0xFULL << (32 + 4 * p)));
    f |= ((u64)streak << (8 + 8 * p)) | ((u64)pos << (24 + 4 * p)) | ((u64)filled << (32 + 4 * p));
    row[RS_FLAGS] = (int64_t)f;
}

// one block: the games that ended in this iteration, in slot order (the samples' positions come from a block scan, so a
// compacted batch, which keeps its slots' order, writes the same samples in the same places)
__global__ void __launch_bounds__(1024)
k_selfplay_resign_account(const u64 *__restrict__ st, int64_t n, int iter, const int32_t *__restrict__ start_iter,
                          const int64_t *__restrict__ serial, u32 k0, u32 k1, int64_t uid0, const int64_t *__restrict__ slot_ids,
                          double threshold, double probe, int64_t *__restrict__ rs, u64 *__restrict__ counters,
                          double *__restrict__ samples, int64_t cap)
{
    __shared__ int warp_tot[32];
    __shared__ long long base_s;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) base_s = (long long)(counters[4] + counters[5]);
    __syncthreads();
    for (int64_t g0 = 0; g0 < n; g0 += 1024) {
        const int64_t g = g0 + t;
        bool cand = false;
        double sample = 0.0;
        if (g < n) {
            const int status = (int)(st[4 * n + g] >> 56);
            if ((status == CCX_ST_WON_P1 || status == CCX_ST_WON_P2) && start_iter[g] <= iter) {
                int64_t *row = rs + g * CCX_RESIGN_WORDS;
                if (row[RS_SERIAL] != serial[g])                                  // never searched: no value, window +inf
                    resign_slot_init(row, serial[g], k0, k1, (u64)(slot_ids ? slot_ids[g] : uid0 + g), probe);
                const u64 f = (u64)row[RS_FLAGS];
                const int would = (int)((f >> 1) & 3);
                if (f & 1) {
                    atomicAdd(&counters[1], 1ULL);
                    if (would) atomicAdd(&counters[2], 1ULL);
                    if (would == status) atomicAdd(&counters[3], 1ULL);
                }
                if ((f & 1) || threshold <= -1.0) { cand = true; sample = __longlong_as_double(row[RS_WMIN + status - 1]); }
            }
        }
        const unsigned b = __ballot_sync(FULL, cand);
        if (lane == 0) warp_tot[warp] = __popc(b);
        __syncthreads();
        long long at = base_s;
        for (int w = 0; w < warp; w++) at += warp_tot[w];
        at += __popc(b & ((1u << lane) - 1u));
        if (cand) {
            if (at < cap) { samples[at] = sample; atomicAdd(&counters[4], 1ULL); }
            else atomicAdd(&counters[5], 1ULL);
        }
        __syncthreads();
        if (t == 0) { int tot = 0; for (int w = 0; w < 32; w++) tot += warp_tot[w]; base_s += tot; }
        __syncthreads();
    }
}

// ---- K11 trajectory pack: kept records -> board_x (u8 planes), pi_y (float32), v_y (int8) ---------------------
// rows[i] = record index of output row i (compacted by the host with torch.nonzero on the flags).
__global__ void __launch_bounds__(128)
k_traj_pack(const int64_t *__restrict__ rows, int64_t m, const u64 *__restrict__ rec_state, const uint16_t *__restrict__ rec_visits,
            const uint8_t *__restrict__ rec_flag, u64 *__restrict__ out_state, float *__restrict__ pi_y, int8_t *__restrict__ v_y)
{
    int64_t i = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (i >= m) return;
    int64_t rec = rows[i];
    uint8_t f = rec_flag[rec];
    bool det = f & REC_TAU_DET;
    double w[10], sum = 0.0;
#pragma unroll
    for (int q = 0; q < 10; q++) {
        int a = lane + 32 * q;
        double N = a < CCX_NUM_ACTIONS ? (double)rec_visits[rec * CCX_NUM_ACTIONS + a] : 0.0;
        w[q] = det ? pow(N, 100.0) : N;                                   // N ** (1 / tau), MCTS.py:132
        sum += w[q];
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
#pragma unroll
    for (int q = 0; q < 10; q++) { int a = lane + 32 * q; if (a < CCX_NUM_ACTIONS) pi_y[i * CCX_NUM_ACTIONS + a] = (float)(w[q] / sum); }
    if (lane < 5) out_state[lane * m + i] = rec_state[rec * 5 + lane];     // plane-major for ccx_encode
    if (lane == 0) v_y[i] = (f & 0xF) == REC_WIN ? 1 : -1;
}

// improved-policy targets (the Gumbel search): pi float64 -> float32 record row (iter % R) * n + slot, for the searched slots
__global__ void __launch_bounds__(128)
k_selfplay_record_pi(int64_t n, int iter, const double *__restrict__ pi, float *__restrict__ rec_pi, int rec_iters)
{
    const int64_t g = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= n) return;
    float x[10];
    bool any = false;
#pragma unroll
    for (int q = 0; q < 10; q++) {
        const int a = lane + 32 * q;
        x[q] = a < CCX_NUM_ACTIONS ? (float)pi[g * CCX_NUM_ACTIONS + a] : 0.0f;
        any |= x[q] > 0.0f;
    }
    if (!__any_sync(FULL, any)) return;                  // not searched (opening ply, inactive or overflowed tree): no record
    const int64_t rec = (int64_t)(iter % rec_iters) * n + g;
#pragma unroll
    for (int q = 0; q < 10; q++) { const int a = lane + 32 * q; if (a < CCX_NUM_ACTIONS) rec_pi[rec * CCX_NUM_ACTIONS + a] = x[q]; }
}

// k_traj_pack with the policy target read from rec_pi
__global__ void __launch_bounds__(128)
k_traj_pack_pi(const int64_t *__restrict__ rows, int64_t m, const u64 *__restrict__ rec_state, const float *__restrict__ rec_pi,
               const uint8_t *__restrict__ rec_flag, u64 *__restrict__ out_state, float *__restrict__ pi_y, int8_t *__restrict__ v_y)
{
    const int64_t i = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= m) return;
    const int64_t rec = rows[i];
    for (int a = lane; a < CCX_NUM_ACTIONS; a += 32) pi_y[i * CCX_NUM_ACTIONS + a] = rec_pi[rec * CCX_NUM_ACTIONS + a];
    if (lane < 5) out_state[lane * m + i] = rec_state[rec * 5 + lane];
    if (lane == 0) v_y[i] = (rec_flag[rec] & 0xF) == REC_WIN ? 1 : -1;
}

extern "C" {

int ccx_selfplay_record_pi(ccx_handle *h, int64_t n, int32_t iter, const double *pi, float *rec_pi, int32_t rec_iters)
{
    if (!h || n < 0 || rec_iters < 1 || iter < 0 || (n && (!pi || !rec_pi))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_selfplay_record_pi<<<(unsigned)((n + 3) / 4), 128, 0, h->stream>>>(n, iter, pi, rec_pi, rec_iters);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_traj_pack_pi(ccx_handle *h, int64_t m, const int64_t *rows, const uint64_t *rec_state, const float *rec_pi,
                     const uint8_t *rec_flag, uint64_t *out_state, float *pi_y, int8_t *v_y)
{
    if (!h || m < 0 || (m && (!rows || !rec_state || !rec_pi || !rec_flag || !out_state || !pi_y || !v_y))) return CCX_ERR_ARG;
    if (m == 0) return CCX_OK;
    k_traj_pack_pi<<<(unsigned)((m + 3) / 4), 128, 0, h->stream>>>(rows, m, (const u64 *)rec_state, rec_pi, rec_flag,
                                                                  (u64 *)out_state, pi_y, v_y);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_set_slot_ids(ccx_handle *h, const int64_t *slot_ids)
{
    if (!h) return CCX_ERR_ARG;
    h->slot_ids = slot_ids;
    ccx_trees_set_uids(h, slot_ids);
    return CCX_OK;
}

int ccx_gamma_noise(ccx_handle *h, int64_t n, int32_t stride, double alpha, uint64_t seed, uint32_t iter, int64_t uid0,
                    double *out)
{
    if (!h || n < 0 || stride < 1 || !(alpha > 0.0) || (n && !out)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    int64_t t = n * stride;
    k_gamma_noise<<<(unsigned)((t + 127) / 128), 128, 0, h->stream>>>(out, n, stride, alpha, (u32)seed, (u32)(seed >> 32), iter, uid0, h->slot_ids);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_selfplay_advance(ccx_handle *h, int64_t n, uint64_t *state, const uint32_t *visits, const int32_t *tree_nodes,
                         uint64_t seed, int32_t iter, int64_t uid0, const int64_t *serial, int64_t total_slots,
                         int32_t random_plies, int32_t tau_switch, int32_t move_limit, uint64_t *rec_state,
                         uint16_t *rec_visits, uint8_t *rec_flag, int32_t rec_iters, uint64_t *counters, uint32_t *move_log)
{
    if (!h || n < 0 || rec_iters < 1 || iter < 0 ||
        (n && (!state || !visits || !tree_nodes || !serial || !rec_state || !rec_visits || !rec_flag || !counters)))
        return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_selfplay_advance<<<(unsigned)((n + SP_WARPS - 1) / SP_WARPS), 32 * SP_WARPS, 0, h->stream>>>(
        (u64 *)state, n, visits, tree_nodes, (u32)seed, (u32)(seed >> 32), iter, uid0, serial, total_slots, random_plies,
        tau_switch, move_limit, (u64 *)rec_state, rec_visits, rec_flag, rec_iters, (u64 *)counters, move_log, h->jump_table, h->slot_ids);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_selfplay_finish(ccx_handle *h, int64_t n, uint64_t *state, int32_t iter, int32_t *start_iter, int64_t *serial,
                        const uint64_t *rec_state, uint8_t *rec_flag, int32_t rec_iters, int32_t max_game_iters, int32_t restart,
                        int64_t *starts_left, uint64_t *counters)
{
    if (!h || n < 0 || rec_iters < 1 || iter < 0 || (n && (!state || !start_iter || !serial || !rec_state || !rec_flag || !counters)))
        return CCX_ERR_ARG;
    if (max_game_iters > rec_iters) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_selfplay_finish<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((u64 *)state, n, iter, start_iter, serial,
                                                                         (const u64 *)rec_state, rec_flag, rec_iters, max_game_iters,
                                                                         restart, (long long *)starts_left, (u64 *)counters);
    CCX_LAUNCHED(h);
    if (restart && starts_left) {
        k_selfplay_restart<<<1, 1024, 0, h->stream>>>((u64 *)state, n, iter, start_iter, serial, (long long *)starts_left);
        CCX_LAUNCHED(h);
    }
    return CCX_OK;
}

int ccx_game_advance(ccx_handle *h, int64_t n, uint64_t *state, const uint32_t *visits, const int32_t *tree_nodes, uint64_t seed,
                     int64_t uid0, double tau, int32_t tau0_after, int32_t move_limit, uint64_t *counters)
{
    if (!h || n < 0 || !(tau > 0.0) || (n && (!state || !counters))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_game_advance<<<(unsigned)((n + SP_WARPS - 1) / SP_WARPS), 32 * SP_WARPS, 0, h->stream>>>((u64 *)state, n, visits, tree_nodes, (u32)seed,
                                                                                              (u32)(seed >> 32), uid0, tau, tau0_after,
                                                                                              move_limit, (u64 *)counters, h->jump_table);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_traj_pack(ccx_handle *h, int64_t m, const int64_t *rows, const uint64_t *rec_state, const uint16_t *rec_visits,
                  const uint8_t *rec_flag, uint64_t *out_state, float *pi_y, int8_t *v_y)
{
    if (!h || m < 0 || (m && (!rows || !rec_state || !rec_visits || !rec_flag || !out_state || !pi_y || !v_y))) return CCX_ERR_ARG;
    if (m == 0) return CCX_OK;
    k_traj_pack<<<(unsigned)((m + 3) / 4), 128, 0, h->stream>>>(rows, m, (const u64 *)rec_state, rec_visits, rec_flag,
                                                               (u64 *)out_state, pi_y, v_y);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_selfplay_resign(ccx_handle *h, int64_t n, uint64_t *state, uint64_t seed, int64_t uid0, const int64_t *serial,
                        double threshold, int32_t plies, double probe, int64_t *resign_state, double *value_out, uint64_t *counters)
{
    if (!h || n < 0 || plies < 1 || plies > CCX_RESIGN_MAX_PLIES || threshold != threshold || probe != probe ||
        (n && (!state || !serial || !resign_state || !counters)))
        return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    ccx_root_view tv;
    const int rc = ccx_trees_root_view(h, &tv);
    if (rc != CCX_OK) return rc;
    if (n > tv.cap_trees) return CCX_ERR_ARG;
    k_selfplay_resign<<<(unsigned)((n + SP_WARPS - 1) / SP_WARPS), 32 * SP_WARPS, 0, h->stream>>>(
        tv, (u64 *)state, n, (u32)seed, (u32)(seed >> 32), uid0, h->slot_ids, serial, threshold, plies, probe, resign_state, value_out,
        (u64 *)counters);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_selfplay_resign_account(ccx_handle *h, int64_t n, const uint64_t *state, int32_t iter, const int32_t *start_iter,
                                const int64_t *serial, uint64_t seed, int64_t uid0, double threshold, double probe,
                                int64_t *resign_state, uint64_t *counters, double *samples, int64_t sample_cap)
{
    if (!h || n < 0 || iter < 0 || sample_cap < 0 || threshold != threshold || probe != probe ||
        (n && (!state || !start_iter || !serial || !resign_state || !counters)) || (sample_cap && !samples))
        return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_selfplay_resign_account<<<1, 1024, 0, h->stream>>>((const u64 *)state, n, iter, start_iter, serial, (u32)seed, (u32)(seed >> 32),
                                                         uid0, h->slot_ids, threshold, probe, resign_state, (u64 *)counters, samples,
                                                         sample_cap);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_selfplay_playout_cap(ccx_handle *h, int64_t n, const uint64_t *state, uint64_t seed, int64_t uid0, const int64_t *serial,
                             int32_t min_ply, double p, int32_t full_budget, int32_t fast_budget, int32_t *budget, uint64_t *counters,
                             uint8_t *keep)
{
    if (!h || n < 0 || !(p >= 0.0 && p <= 1.0) || fast_budget < 0 || fast_budget > full_budget ||
        (n && (!state || !serial || !budget || !counters)))
        return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_selfplay_playout_cap<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((const u64 *)state, n, (u32)seed, (u32)(seed >> 32), uid0,
                                                                              h->slot_ids, serial, min_ply, p, full_budget, fast_budget,
                                                                              budget, (u64 *)counters, keep);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

}  // extern "C"
