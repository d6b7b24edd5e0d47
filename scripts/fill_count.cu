// fill_count.cu — host build of the random-legal ply (pick_first_start / fill_step / pick_first_to in
// chinesecheckersagent_b200/csrc/ccx_device.cuh, stepped the way the step kernels step a game) that records how many fill
// steps the picked checker's jump closure costs at every game-ply.  Loaded by scripts/fill_model.py; never linked into
// libccx.so.
#include "../chinesecheckersagent_b200/csrc/ccx_device.cuh"

static TriTables host_tables()
{
    static uint8_t T3[CCX_JT3_BYTES] __attribute__((aligned(16)));
    static u64 NB[64], CI[64], O[64], OT[64], OD[64];
    build_jump_table3(T3, 0, 1);
    for (int q = 0; q < 64; q++) {                   // as tri_tables_load in ccx_env.cu
        const bool on = (CCX_VALID >> q) & 1;
        NB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
        CI[q] = on ? tri_cell_info(q) : 0ULL;
        O[q] = 1ULL << q;
        OT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
        OD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
    }
    TriTables t = {T3, NB, CI, O, OT, OD};
    return t;
}

extern "C" {

// n games from the start position (game ids 0..n-1), `plies` random plies; E[i * (plies - warm) + t - warm] = fill steps of game
// i at ply t >= warm (0 for a ply that passes).  Returns the walk-test expansions (checkers without an empty neighbour) summed
// over the recorded game-plies.
long long fc_count(int n, int plies, int warm, uint64_t seed, uint8_t *E)
{
    const TriTables T = host_tables();
    const int P = plies - warm;
    long long nowalk = 0;
    for (int i = 0; i < n; i++) {
        Game g;
        reset_start(g);
        u64 occT_all, occD_all;
        tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all);
        for (int t = 0; t < plies; t++) {
            const Philox4 rnd = philox4x32_10((u32)seed, (u32)(seed >> 32), (u32)t, 0u, (u32)i, 0u);
            if (t >= warm) nowalk += 6 - ccx_popc(walk_movable(g.occ_me, g.occ_me | g.occ_op, g.cells_me));
            int from, steps = 0;
            JumpFill f;
            const int id = pick_first_start(g, occT_all, occD_all, rnd.x, T, from, f);
            if (id >= 0) {
                while (f.todo) { fill_step(f, T); steps++; }
                const int to = pick_first_to(g.occ_me | g.occ_op, from, f, rnd.y, T);
                apply_move(g, id, from, to);
                occT_all ^= T.sOT[from] | T.sOT[to];
                occD_all ^= T.sOD[from] | T.sOD[to];
                if (winner_of(g)) { reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
            }
            if (t >= warm) E[(size_t)i * P + (t - warm)] = (uint8_t)(steps < 255 ? steps : 255);
        }
    }
    return nowalk;
}

}  // extern "C"
