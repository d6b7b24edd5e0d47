// carry_ply.cu — TEST-ONLY host instantiation of k_step_random_carry's ply (carry_ply_start / fill_step / carry_ply_to and
// the selects in chinesecheckersagent_b200/csrc/ccx_device.cuh), stepped the way the kernel steps one game, so that the CPU
// test-suite runs the kernel's own source against the oracle and against select64.  Never linked into libccx.so.
#include "../../chinesecheckersagent_b200/csrc/ccx_device.cuh"
#include "../../include/ccx.h"

static TriTables host_tables()
{
    static uint8_t T3[CCX_JT3_BYTES] __attribute__((aligned(16)));
    static u64 NB[64], CI[64], O[64], OT[64], OD[64];
    static u32 SEL[128];
    static bool built = false;
    if (!built) {
        build_jump_table3(T3, 0, 1);
        for (int q = 0; q < 64; q++) {               // as tri_tables_load<TPB, true> in ccx_env.cu
            const bool on = (CCX_VALID >> q) & 1;
            NB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
            CI[q] = on ? tri_cell_info(q) : 0ULL;
            O[q] = 1ULL << q;
            OT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
            OD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
        }
        for (u32 q = 0; q < 128; q++) SEL[q] = sel7_entry(q);
        built = true;
    }
    TriTables t = {T3, NB, CI, O, OT, OD, SEL};
    return t;
}

extern "C" {

// fast[i] = select64_step(m[i], k[i]), ref[i] = select64(m[i], k[i]); requires k[i] < popc(m[i])
void cp_select64(const u64 *m, const u32 *k, int64_t n, int32_t *fast, int32_t *ref)
{
    const TriTables T = host_tables();
    for (int64_t i = 0; i < n; i++) {
        fast[i] = select64_step(m[i], k[i], T.sSel);
        ref[i] = select64(m[i], k[i]);
    }
}

// out[v * 7 + r] = sel7_rank(v, r) for every 7-bit value v and rank r < 7 (-1 where r >= popc(v))
void cp_sel7(int32_t *out)
{
    const TriTables T = host_tables();
    for (u32 v = 0; v < 128; v++)
        for (u32 r = 0; r < 7; r++) out[v * 7 + r] = r < (u32)ccx_popc(v) ? (int32_t)sel7_rank(T.sSel, v, r) : -1;
}

// ccx_step_random on the host with the carry kernel's ply: state words 0-4 in place, wins[2] accumulated, trace rows as the
// kernel writes them.  The occupancy in the T / D layouts is carried through the fill the way the kernel carries it.
void cp_step_random(u64 *st, int64_t n, int64_t gid0, uint64_t seed, uint32_t step0, int plies, u64 *wins, u64 *trace,
                    int64_t trace_games)
{
    const TriTables T = host_tables();
    const u32 k0 = (u32)seed, k1 = (u32)(seed >> 32);
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
            const Philox4 rnd = philox4x32_10(k0, k1, step0 + (u32)t, 0u, (u32)gid, (u32)(gid >> 32));
            int from;
            JumpFill f;
            const int id = carry_ply_start(g, occT_all, occD_all, rnd.x, T, from, f);
            if (id < 0) continue;
            while (f.todo) fill_step(f, T);
            const int to = carry_ply_to(f, rnd.y, T);
            apply_move(g, id, from, to);
            occT_all = f.occT | T.sOT[to];
            occD_all = f.occD | T.sOD[to];
            const int win = winner_of(g);
            if (row) row[11] = (u64)from | ((u64)to << 8) | ((u64)win << 16) | ((u64)id << 24);
            if (win) { wins[win - 1]++; reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
        }
        bool p2 = (g.meta >> 48) & 1;
        st[0 * n + i] = p2 ? g.occ_op : g.occ_me; st[1 * n + i] = p2 ? g.occ_me : g.occ_op;
        st[2 * n + i] = p2 ? g.cells_op : g.cells_me; st[3 * n + i] = p2 ? g.cells_me : g.cells_op;
        st[4 * n + i] = g.meta;
    }
}

}  // extern "C"
