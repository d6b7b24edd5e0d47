// pick_first.cu — TEST-ONLY host instantiation of the pick-first random ply (pick_random_first and the three-layout helpers
// in chinesecheckersagent_b200/csrc/ccx_device.cuh), stepped the way k_step_random_pick steps a game, so that the CPU
// test-suite runs the kernel's own source against the oracle.  Never linked into libccx.so.
#include "../../chinesecheckersagent_b200/csrc/ccx_device.cuh"
#include "../../include/ccx.h"

static TriTables host_tables()
{
    static uint8_t T3[CCX_JT3_BYTES] __attribute__((aligned(16)));
    static u64 NB[64], CI[64], O[64], OT[64], OD[64];
    static bool built = false;
    if (!built) {
        build_jump_table3(T3, 0, 1);
        for (int q = 0; q < 64; q++) {               // as tri_tables_load in ccx_env.cu
            const bool on = (CCX_VALID >> q) & 1;
            NB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
            CI[q] = on ? tri_cell_info(q) : 0ULL;
            O[q] = 1ULL << q;
            OT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
            OD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
        }
        built = true;
    }
    TriTables t = {T3, NB, CI, O, OT, OD};
    return t;
}

extern "C" {

// ccx_step_random on the host: state words 0-4 in place, wins[2] accumulated, trace rows as the kernel writes them
void pf_step_random(u64 *st, int64_t n, int64_t gid0, uint64_t seed, uint32_t step0, int plies, u64 *wins, u64 *trace,
                    int64_t trace_games)
{
    const TriTables T = host_tables();
    for (int64_t i = 0; i < n; i++) {
        Game g;
        {
            u64 occ1 = st[0 * n + i], occ2 = st[1 * n + i], c1 = st[2 * n + i], c2 = st[3 * n + i];
            g.meta = st[4 * n + i];
            bool p2 = (g.meta >> 48) & 1;
            g.occ_me = p2 ? occ2 : occ1; g.occ_op = p2 ? occ1 : occ2;
            g.cells_me = p2 ? c2 : c1;   g.cells_op = p2 ? c1 : c2;
        }
        const u64 gid = (u64)(gid0 + i);
        u64 occT_all, occD_all;
        tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all);
        for (int t = 0; t < plies; t++) {
            u64 *row = nullptr;
            if (trace && i < trace_games) {
                row = trace + ((int64_t)t * trace_games + i) * CCX_TRACE_WORDS;
                u64 dest[6];
                movegen_tri(g.occ_me | g.occ_op, occT_all, occD_all, g.cells_me, dest, T);
                bool p2 = (g.meta >> 48) & 1;
                row[0] = p2 ? g.occ_op : g.occ_me; row[1] = p2 ? g.occ_me : g.occ_op;
                row[2] = p2 ? g.cells_op : g.cells_me; row[3] = p2 ? g.cells_me : g.cells_op;
                row[4] = g.meta & 0x00FFFFFFFFFFFFFFULL;
                for (int q = 0; q < 6; q++) row[5 + q] = dest[q];
                row[11] = 0xFFULL | (0xFFULL << 8) | (0xFFULL << 24);
            }
            Philox4 rnd = philox4x32_10((u32)seed, (u32)(seed >> 32), step0 + (u32)t, 0u, (u32)gid, (u32)(gid >> 32));
            int from, to;
            const int pid = pick_random_first(g, occT_all, occD_all, rnd.x, rnd.y, T, from, to);
            if (pid < 0) continue;
            apply_move(g, pid, from, to);
            occT_all ^= T.sOT[from] | T.sOT[to];
            occD_all ^= T.sOD[from] | T.sOD[to];
            const int win = winner_of(g);
            if (row) row[11] = (u64)from | ((u64)to << 8) | ((u64)win << 16) | ((u64)pid << 24);
            if (win) { wins[win - 1]++; reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
        }
        bool p2 = (g.meta >> 48) & 1;
        st[0 * n + i] = p2 ? g.occ_op : g.occ_me; st[1 * n + i] = p2 ? g.occ_me : g.occ_op;
        st[2 * n + i] = p2 ? g.cells_op : g.cells_me; st[3 * n + i] = p2 ? g.cells_me : g.cells_op;
        st[4 * n + i] = g.meta;
    }
}

}  // extern "C"
