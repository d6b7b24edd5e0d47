// fill_latency.cu — microbenchmark of the jump flood fill alone: the fill k_step_random_carry ran before its per-cell
// constants were computed with ALU instructions (fill_start with the walk seed, then fill_step: FLO + one tri_cell_info load
// per step) against the one it runs now (carry_fill_start, which takes the first step, then fill_step_carry), on fill start
// states recorded from the host model of the random-legal ply.  Every lane runs S fills one after the other, the warp each
// as long as its longest lane (lockstep), so clock64 over the loop divided by the warp's fill iterations is the cost of one
// step with that many warps per SM to hide its latency.  Loaded by scripts/fill_latency.py; never linked into libccx.so.
#include "../chinesecheckersagent_b200/csrc/ccx_device.cuh"

#define FL_TPB 448

static __host__ __device__ void cell_tables(u64 *NB, u64 *CI, u64 *O, u64 *OT, u64 *OD)
{
    for (int q = 0; q < 64; q++) {                   // as tri_tables_load in ccx_env.cu
        const bool on = (CCX_VALID >> q) & 1;
        NB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
        CI[q] = on ? tri_cell_info(q) : 0ULL;
        O[q] = 1ULL << q;
        OT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
        OD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
    }
}

// NEW = 0: the fill before this change, NEW = 1: the fill k_step_random_carry runs.  MINB 2 so that one build runs at one
// and at two 448-lane blocks per SM (14 and 28 warps).
template <bool NEW>
__global__ void __launch_bounds__(FL_TPB, 2, 1)
k_fill(const u64 *__restrict__ st, int64_t nstates, int S, const uint8_t *__restrict__ jt3, long long *__restrict__ cyc,
       unsigned *__restrict__ iters, u64 *__restrict__ sum)
{
    __shared__ __align__(16) uint8_t sAll[CCX_JT3_BYTES + 5 * 64 * 8];
    u64 *sNB = reinterpret_cast<u64 *>(sAll + CCX_JT3_BYTES), *sCI = sNB + 64, *sO = sNB + 128, *sOT = sNB + 192, *sOD = sNB + 256;
    for (int q = threadIdx.x; q < CCX_JT3_BYTES / 16; q += FL_TPB) reinterpret_cast<uint4 *>(sAll)[q] = reinterpret_cast<const uint4 *>(jt3)[q];
    if (threadIdx.x == 0) cell_tables(sNB, sCI, sO, sOT, sOD);
    __syncthreads();
    const TriTables T = {sAll, sNB, sCI, sO, sOT, sOD, nullptr};
    const int lanes = gridDim.x * FL_TPB, i = blockIdx.x * FL_TPB + threadIdx.x;
    // state s of lane i: (i + s * lanes) mod nstates (> lanes), so consecutive lanes read consecutive states; [4][nstates]:
    // occupancy, T and D layouts, origin
    int idx = i;
    u64 occ = st[idx], occT = st[nstates + idx], occD = st[2 * nstates + idx];
    int from = (int)st[3 * nstates + idx];
    u64 acc = 0;
    unsigned it = 0;
    const long long t0 = clock64();
    for (int s = 0; s < S; s++) {
        idx += lanes;                                 // the next state's loads are in flight during this fill
        if (idx >= nstates) idx -= (int)nstates;
        const u64 n_occ = st[idx], n_occT = st[nstates + idx], n_occD = st[2 * nstates + idx];
        const int n_from = (int)st[3 * nstates + idx];
        JumpFill f;
        unsigned steps;
        if (NEW) {
            f = carry_fill_start(from, occ, occT, occD, T);
            steps = 1;
            while (f.todo) { fill_step_carry(f, T.sT); steps++; }
        } else {
            f = fill_start(from, occ, occT, occD, T);
            f.reach = T.sNB[from] & ~occ;
            steps = 0;
            while (f.todo) { fill_step(f, T); steps++; }
        }
        acc += f.reach * (u64)(2 * s + 1);
        it += __reduce_max_sync(0xFFFFFFFFu, steps);
        occ = n_occ; occT = n_occT; occD = n_occD; from = n_from;
    }
    const long long t1 = clock64();
    if ((threadIdx.x & 31) == 0) { cyc[i >> 5] = t1 - t0; iters[i >> 5] = it; }
    sum[i] = acc;
}

extern "C" {

int64_t fl_table_bytes() { return CCX_JT3_BYTES; }

void fl_table(uint8_t *T3) { build_jump_table3(T3, 0, 1); }     // T3: fl_table_bytes() bytes

// n games from the start position (game ids 0..n-1), `plies` random plies as the step kernels play them; the fill start state
// of every ply t >= warm that moves goes to st ([4][capacity]: occupancy, T / D layouts, origin).  Returns the states recorded.
int64_t fl_record(int n, int plies, int warm, uint64_t seed, u64 *st, int64_t capacity)
{
    static uint8_t T3[CCX_JT3_BYTES] __attribute__((aligned(16)));
    static u64 NB[64], CI[64], O[64], OT[64], OD[64];
    build_jump_table3(T3, 0, 1);
    cell_tables(NB, CI, O, OT, OD);
    const TriTables T = {T3, NB, CI, O, OT, OD, nullptr};
    int64_t m = 0;
    for (int i = 0; i < n && m < capacity; i++) {
        Game g;
        reset_start(g);
        u64 occT_all, occD_all;
        tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all);
        for (int t = 0; t < plies && m < capacity; t++) {
            const Philox4 rnd = philox4x32_10((u32)seed, (u32)(seed >> 32), (u32)t, 0u, (u32)i, 0u);
            int from;
            JumpFill f;
            const int id = pick_first_start(g, occT_all, occD_all, rnd.x, T, from, f);
            if (id < 0) continue;
            if (t >= warm) {
                st[m] = g.occ_me | g.occ_op; st[capacity + m] = occT_all; st[2 * capacity + m] = occD_all; st[3 * capacity + m] = (u64)from;
                m++;
            }
            while (f.todo) fill_step(f, T);
            const int to = pick_first_to(g.occ_me | g.occ_op, from, f, rnd.y, T);
            apply_move(g, id, from, to);
            occT_all ^= T.sOT[from] | T.sOT[to];
            occD_all ^= T.sOD[from] | T.sOD[to];
            if (winner_of(g)) { reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
        }
    }
    return m;
}

// one launch of k_fill<is_new> with `blocks` 448-lane blocks on the legacy default stream; returns the launch error
int fl_run(int is_new, int blocks, const u64 *st, int64_t nstates, int S, const uint8_t *jt3, long long *cyc, unsigned *iters, u64 *sum)
{
    if (is_new) k_fill<true><<<blocks, FL_TPB>>>(st, nstates, S, jt3, cyc, iters, sum);
    else k_fill<false><<<blocks, FL_TPB>>>(st, nstates, S, jt3, cyc, iters, sum);
    return (int)cudaGetLastError();
}

}  // extern "C"
