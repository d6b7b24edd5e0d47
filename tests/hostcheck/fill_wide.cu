// fill_wide.cu — TEST-ONLY host instantiation of the one-wave carry kernel's wide answer tables (build_jump_table_wide and
// the expansion over them in chinesecheckersagent_b200/csrc/ccx_device.cuh) next to build_jump_table3's tables and the fill
// the other kernels run, so that the CPU test-suite compares the two on the kernel's own source.  Never linked into libccx.so.
#include "../../chinesecheckersagent_b200/csrc/ccx_device.cuh"

static uint8_t T3[CCX_JT3_BYTES] __attribute__((aligned(16)));
static u64 W[CCX_JTW_BYTES / 8];

static TriTables host_tables()
{
    static u64 NB[64], CI[64], O[64], OT[64], OD[64];
    static bool built = false;
    if (!built) {
        build_jump_table3(T3, 0, 1);
        build_jump_table_wide(W, T3, 0, 1);
        for (int q = 0; q < 64; q++) {               // as tri_tables_load / wide_tables_load in ccx_env.cu
            const bool on = (CCX_VALID >> q) & 1;
            NB[q] = on ? (neighbours(1ULL << q) & CCX_VALID) : 0ULL;
            CI[q] = on ? tri_cell_info(q) : 0ULL;
            O[q] = 1ULL << q;
            OT[q] = on ? 1ULL << tri_tbit(q) : 0ULL;
            OD[q] = on ? 1ULL << tri_dbit(q) : 0ULL;
        }
        built = true;
    }
    TriTables t = {T3, NB, CI, O, OT, OD, nullptr, W};
    return t;
}

extern "C" {

int64_t fw_jt3_bytes() { return CCX_JT3_BYTES; }
int64_t fw_wide_words() { return CCX_JTW_BYTES / 8; }

// copies of both table sets as the kernels receive them
void fw_tables(uint8_t *t3, u64 *w)
{
    host_tables();
    for (int i = 0; i < CCX_JT3_BYTES; i++) t3[i] = T3[i];
    for (int i = 0; i < CCX_JTW_BYTES / 8; i++) w[i] = W[i];
}

// For every occupancy occ[i] (on-board cells) and every on-board cell c of mover[i] (the mover is added to the occupancy):
// the destination set of the fill the other kernels run (walks | fill_start + fill_step until done) and of the one-wave carry
// kernel's (carry_fill_start<true> + fill_step_carry over the wide tables until done).  Returns the number of pairs where
// they differ, or where a single expansion differs (the wide one against expand_cell_tri, on the mover-free words of every
// expanded cell and on the full ones for the origin); *pairs counts all pairs, *steps the expansions compared.
int64_t fw_closures(const u64 *occ, const u64 *mover, int64_t n, int64_t *pairs, int64_t *steps)
{
    const TriTables T = host_tables();
    int64_t bad = 0, cnt = 0, nst = 0;
    for (int64_t i = 0; i < n; i++) {
        u64 m = mover[i] & CCX_VALID;
        while (m) {
            const int c = 63 - ccx_clzll(m);
            m ^= 1ULL << c;
            const u64 occ_all = (occ[i] & CCX_VALID) | (1ULL << c);
            u64 occT_all = 0, occD_all = 0;
            for (int q = 0; q < 64; q++)
                if ((occ_all >> q) & 1) { occT_all |= T.sOT[q]; occD_all |= T.sOD[q]; }
            if (expand_cell_carry(c, occ_all, occT_all, occD_all, T.sW) != expand_cell_tri(c, occ_all, occT_all, occD_all, T.sT, T.sCI)) bad++;
            JumpFill a = fill_start(c, occ_all, occT_all, occD_all, T);
            while (a.todo) {
                const int e = 63 - ccx_clzll(a.todo);
                if (expand_cell_carry(e, a.occ, a.occT, a.occD, T.sW) != expand_cell_tri(e, a.occ, a.occT, a.occD, T.sT, T.sCI)) bad++;
                nst++;
                fill_step(a, T);
            }
            const u64 want = (T.sNB[c] & ~occ_all) | a.reach;
            JumpFill b = carry_fill_start<true>(c, occ_all, occT_all, occD_all, T);
            while (b.todo) fill_step_carry(b, T.sW);
            if (b.reach != want || b.o != a.o || b.occ != a.occ || b.occT != a.occT || b.occD != a.occD) bad++;
            cnt++;
        }
    }
    *pairs = cnt;
    *steps = nst;
    return bad;
}

// the TRACE rows' move generation: movegen_tri over the wide tables against movegen_tri over build_jump_table3's, for the
// side to move (occ_me, cells_me) of every position; returns the number of positions whose six sets differ
int64_t fw_movegen(const u64 *occ_me, const u64 *occ_op, const u64 *cells_me, int64_t n)
{
    const TriTables T = host_tables();
    int64_t bad = 0;
    for (int64_t i = 0; i < n; i++) {
        const u64 occ_all = occ_me[i] | occ_op[i];
        u64 occT_all = 0, occD_all = 0;
        for (int q = 0; q < 64; q++)
            if ((occ_all >> q) & 1) { occT_all |= T.sOT[q]; occD_all |= T.sOD[q]; }
        u64 a[6], b[6];
        movegen_tri(occ_all, occT_all, occD_all, cells_me[i], a, T);
        movegen_tri<true>(occ_all, occT_all, occD_all, cells_me[i], b, T);
        for (int k = 0; k < 6; k++) bad += a[k] != b[k];
    }
    return bad;
}

}  // extern "C"
