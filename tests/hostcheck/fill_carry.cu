// fill_carry.cu — TEST-ONLY host instantiation of k_step_random_carry's fill (carry_cell, carry_fill_start, fill_step_carry in
// chinesecheckersagent_b200/csrc/ccx_device.cuh) next to the fill the other kernels run (tri_cell_info, fill_start,
// fill_step), so that the CPU test-suite compares the two on the kernel's own source.  Never linked into libccx.so.
#include "../../chinesecheckersagent_b200/csrc/ccx_device.cuh"

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
    TriTables t = {T3, NB, CI, O, OT, OD, nullptr};
    return t;
}

extern "C" {

// out[c * 7 + ...] for every cell c < 64: tri_cell_info(c) (lo, hi), then carry_cell(c) (rsel, csel, dsel, lp8, sh)
void fc_cell_info(uint64_t *out)
{
    for (int c = 0; c < 64; c++) {
        const u64 ci = tri_cell_info(c);
        const CarryCell q = carry_cell(c);
        uint64_t *o = out + c * 7;
        o[0] = (u32)ci; o[1] = (u32)(ci >> 32);
        o[2] = q.rsel; o[3] = q.csel; o[4] = q.dsel; o[5] = q.lp8; o[6] = q.sh;
    }
}

// PRMT as the host model computes it (ccx_byte_of): out[i] = prmt(lo[i], hi[i], sel[i])
void fc_prmt(const u32 *lo, const u32 *hi, const u32 *sel, int64_t n, u32 *out)
{
    for (int64_t i = 0; i < n; i++) out[i] = ccx_byte_of(lo[i], hi[i], sel[i]);
}

// the diagonal answer the carry step reads for cell c when the D-layout occupancy is occD (used on the corner cells, whose
// selector picks a zero byte): 8 bytes of T3 at the answer column
uint64_t fc_diag_answer(int c, uint64_t occD)
{
    const TriTables T = host_tables();
    const CarryCell q = carry_cell(c);
    const u32 dia7 = ccx_byte_of((u32)occD, (u32)(occD >> 32), q.dsel);
    return *reinterpret_cast<const u64 *>(T.sT + CCX_JT3_DIA + dia7 * (CCX_JT3_NLP * 8) + q.lp8);
}

// For every occupancy occ[i] (on-board cells) and every on-board cell c of mover[i] (the mover is added to the occupancy):
// the destination set of the fill the other kernels run (walks | fill_start + fill_step until done) and of the carry kernel's
// (carry_fill_start + fill_step_carry until done).  Returns the number of (occupancy, cell) pairs where they differ, or where
// a single expansion differs (expand_cell_carry against expand_cell_tri, on the mover-free words and, for the origin, on the
// full ones); *pairs counts all pairs.
int64_t fc_closures(const u64 *occ, const u64 *mover, int64_t n, int64_t *pairs)
{
    const TriTables T = host_tables();
    int64_t bad = 0, cnt = 0;
    for (int64_t i = 0; i < n; i++) {
        u64 m = mover[i] & CCX_VALID;
        while (m) {
            const int c = 63 - ccx_clzll(m);
            m ^= 1ULL << c;
            const u64 occ_all = (occ[i] & CCX_VALID) | (1ULL << c);
            u64 occT_all = 0, occD_all = 0;
            for (int q = 0; q < 64; q++)
                if ((occ_all >> q) & 1) { occT_all |= T.sOT[q]; occD_all |= T.sOD[q]; }
            JumpFill a = fill_start(c, occ_all, occT_all, occD_all, T);
            while (a.todo) {
                const int e = 63 - ccx_clzll(a.todo);
                if (expand_cell_carry(e, a.occ, a.occT, a.occD, T.sT) != expand_cell_tri(e, a.occ, a.occT, a.occD, T.sT, T.sCI)) bad++;
                fill_step(a, T);
            }
            const u64 want = (T.sNB[c] & ~occ_all) | a.reach;
            JumpFill b = carry_fill_start(c, occ_all, occT_all, occD_all, T);
            if (b.todo != expand_cell_tri(c, a.occ, a.occT, a.occD, T.sT, T.sCI)) bad++;
            while (b.todo) fill_step_carry(b, T.sT);
            if (b.reach != want || b.o != a.o || b.occ != a.occ || b.occT != a.occT || b.occD != a.occD) bad++;
            cnt++;
        }
    }
    *pairs = cnt;
    return bad;
}

}  // extern "C"
