// spec_pick.cu — TEST-ONLY host instantiation of the carry kernel's speculative ply start (carry_ply_start in
// chinesecheckersagent_b200/csrc/ccx_device.cuh), checked position by position against pick_first_start and against the exact
// pick it replaces (walk bits, no-walk expansions, rank table, written out below), on both table sets.  Never linked into
// libccx.so.
#include "../../chinesecheckersagent_b200/csrc/ccx_device.cuh"

static uint8_t T3[CCX_JT3_BYTES] __attribute__((aligned(16)));
static u64 W[CCX_JTW_BYTES / 8];

static TriTables host_tables()
{
    static u64 NB[64], CI[64], O[64], OT[64], OD[64];
    static u32 SEL[128];
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
        for (u32 q = 0; q < 128; q++) SEL[q] = sel7_entry(q);
        built = true;
    }
    TriTables t = {T3, NB, CI, O, OT, OD, SEL, W};
    return t;
}

// the ply start without speculation: the movable set from the walk bits and one expansion per checker without a walk, the
// checker by the rank table, then carry_fill_start
template <bool WIDE>
static int exact_ply_start(const Game &g, u64 occT_all, u64 occD_all, u32 r0, const TriTables &T, int &from, JumpFill &f,
                           u32 &walks, u32 &movable)
{
    const u64 occ_all = g.occ_me | g.occ_op;
    walks = movable = walk_movable(g.occ_me, occ_all, g.cells_me);
    for (int k = 0; k < 6; k++)
        if (!((movable >> k) & 1) &&
            expand_cell_carry((int)((g.cells_me >> (8 * k)) & 0x3F), occ_all, occT_all, occD_all, carry_tables<WIDE>(T)))
            movable |= 1u << k;
    if (!movable) return -1;
    const int id = (int)sel7_rank(T.sSel, movable, ccx_umulhi(r0, (u32)ccx_popc(movable)));
    from = (int)((g.cells_me >> (8 * id)) & 0x3F);
    f = carry_fill_start<WIDE>(from, occ_all, occT_all, occD_all, T);
    return id;
}

static bool same_fill(const JumpFill &a, const JumpFill &b)
{
    return a.o == b.o && a.occ == b.occ && a.occT == b.occT && a.occD == b.occD && a.todo == b.todo && a.reach == b.reach;
}

// compares the three starts at one position; returns the number of disagreements.  walks / movable: the exact reference's
// checkers with a walk and checkers that can move (bit k = checker k), independent of the code under test.
template <bool WIDE>
static int64_t check_position(const Game &g, u64 occT_all, u64 occD_all, u32 r0, const TriTables &T, int &id_out,
                              int &from_out, JumpFill &f_out, u32 &walks, u32 &movable)
{
    int64_t bad = 0;
    int from_s = -1, from_e = -1, from_p = -1;
    JumpFill fs = {}, fe = {}, fp = {};
    const int ids = carry_ply_start<WIDE>(g, occT_all, occD_all, r0, T, from_s, fs);
    const int ide = exact_ply_start<WIDE>(g, occT_all, occD_all, r0, T, from_e, fe, walks, movable);
    const int idp = pick_first_start(g, occT_all, occD_all, r0, T, from_p, fp);
    if (ids != ide || ids != idp) bad++;
    if (ids >= 0) {
        if (from_s != from_e || from_s != from_p || !same_fill(fs, fe)) bad++;
        JumpFill a = fs;                              // the whole destination set: the carry fill's reach after the last
        while (a.todo) fill_step_carry(a, carry_tables<WIDE>(T));         // step, the pick kernel's walks | closure
        while (fp.todo) fill_step(fp, T);
        if (a.reach != ((T.sNB[from_p] & ~(g.occ_me | g.occ_op)) | fp.reach)) bad++;
    }
    id_out = ids; from_out = from_s; f_out = fs;
    return bad;
}

extern "C" {

// Steps n games `plies` plies with the carry kernel's ply (carry_ply_start, fill_step_carry, carry_ply_to, apply_move,
// win / reset) on the wide tables (wide != 0) or build_jump_table3's and checks every ply start against the exact start and
// pick_first_start.  st: state words 0-4 as ccx_step_random takes them, updated in place.  out[0] = disagreements,
// out[1] = ply starts checked, out[2] = starts with a checker without a walk (where carry_ply_start falls back), out[3] =
// passes, out[4] = starts with a checker that cannot move at all; out[2..4] from the exact reference's walk_movable and
// expansions, not from the code under test.
void sp_check(u64 *st, int64_t n, int64_t gid0, uint64_t seed, uint32_t step0, int plies, int wide, int64_t *out)
{
    const TriTables T = host_tables();
    const u32 k0 = (u32)seed, k1 = (u32)(seed >> 32);
    out[0] = out[1] = out[2] = out[3] = out[4] = 0;
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
            const Philox4 rnd = philox4x32_10(k0, k1, step0 + (u32)t, 0u, (u32)gid, (u32)(gid >> 32));
            int id, from;
            JumpFill f;
            u32 walks, movable;
            out[0] += wide ? check_position<true>(g, occT_all, occD_all, rnd.x, T, id, from, f, walks, movable)
                           : check_position<false>(g, occT_all, occD_all, rnd.x, T, id, from, f, walks, movable);
            out[1]++;
            out[2] += walks != 0x3F;
            out[4] += movable != 0x3F;
            if (id < 0) { out[3]++; continue; }
            while (f.todo) {
                if (wide) fill_step_carry(f, T.sW); else fill_step_carry(f, T.sT);
            }
            const int to = carry_ply_to(f, rnd.y, T);
            apply_move(g, id, from, to);
            occT_all = f.occT | T.sOT[to];
            occD_all = f.occD | T.sOD[to];
            if (winner_of(g)) { reset_start(g); tri_build(g.cells_me, g.cells_op, T.sOT, T.sOD, occT_all, occD_all); }
        }
        bool p2 = (g.meta >> 48) & 1;
        st[0 * n + i] = p2 ? g.occ_op : g.occ_me; st[1 * n + i] = p2 ? g.occ_me : g.occ_op;
        st[2 * n + i] = p2 ? g.cells_op : g.cells_me; st[3 * n + i] = p2 ? g.cells_me : g.cells_op;
        st[4 * n + i] = g.meta;
    }
}

// The three starts on n given boards (occupancy words and the mover's cells; the T / D layouts are built from the
// occupancy bits, so a board may hold more than the opponent's six checkers, e.g. every cell but the mover's filled).
// out as in sp_check, with out[1] = n.
void sp_check_boards(const u64 *occ_me, const u64 *occ_op, const u64 *cells_me, const u32 *r0, int64_t n, int wide,
                     int64_t *out)
{
    const TriTables T = host_tables();
    out[0] = out[1] = out[2] = out[3] = out[4] = 0;
    for (int64_t i = 0; i < n; i++) {
        Game g = {occ_me[i], occ_op[i], cells_me[i], 0, 0};
        u64 occT_all = 0, occD_all = 0;
        for (int c = 0; c < 64; c++)
            if (((g.occ_me | g.occ_op) >> c) & 1) { occT_all |= T.sOT[c]; occD_all |= T.sOD[c]; }
        int id, from;
        JumpFill f;
        u32 walks, movable;
        out[0] += wide ? check_position<true>(g, occT_all, occD_all, r0[i], T, id, from, f, walks, movable)
                       : check_position<false>(g, occT_all, occD_all, r0[i], T, id, from, f, walks, movable);
        out[1]++;
        out[2] += walks != 0x3F;
        out[3] += id < 0;
        out[4] += movable != 0x3F;
    }
}

// Exhaustive search: the number of placements of the mover's six checkers that `opponents` opponent checkers can box in so
// that movegen finds no move for any of them.  Every empty neighbour of the mover's checkers must hold an opponent, so only
// placements with at most `opponents` such neighbours are tried, each with every choice of the remaining opponents' cells.
int64_t sp_boxed_in_count(int opponents)
{
    int cells[49], n = 0, a[6];
    for (int c = 0; c < 64; c++) if ((CCX_VALID >> c) & 1) cells[n++] = c;
    int64_t found = 0;
    for (a[0] = 0; a[0] < n; a[0]++) for (a[1] = a[0] + 1; a[1] < n; a[1]++) for (a[2] = a[1] + 1; a[2] < n; a[2]++)
    for (a[3] = a[2] + 1; a[3] < n; a[3]++) for (a[4] = a[3] + 1; a[4] < n; a[4]++) for (a[5] = a[4] + 1; a[5] < n; a[5]++) {
        u64 M = 0, cm = 0;
        for (int k = 0; k < 6; k++) { M |= 1ULL << cells[a[k]]; cm |= (u64)cells[a[k]] << (8 * k); }
        const u64 N = neighbours(M) & CCX_VALID & ~M;
        const int need = opponents - ccx_popcll(N);
        if (need < 0) continue;
        int rest[49], r = 0, b[49];
        for (int q = 0; q < n; q++) if (!(((M | N) >> cells[q]) & 1)) rest[r++] = cells[q];
        if (need > r) continue;
        for (int q = 0; q < need; q++) b[q] = q;
        for (;;) {
            u64 O = N;
            for (int q = 0; q < need; q++) O |= 1ULL << rest[b[q]];
            u64 dest[6];
            movegen(M | O, cm, dest);
            if (!(dest[0] | dest[1] | dest[2] | dest[3] | dest[4] | dest[5])) { found++; break; }
            int q = need - 1;
            while (q >= 0 && b[q] == r - need + q) q--;
            if (q < 0) break;
            b[q]++;
            for (int p = q + 1; p < need; p++) b[p] = b[p - 1] + 1;
        }
    }
    return found;
}

}  // extern "C"
