// ccx_device.cuh — device-side building blocks shared by every kernel: bitboard shifts, long-jump
// flood fill (board.py:139-211), move application (board.py:226-250), win test (board.py:89-111),
// Philox4x32-10.  sm_100a only.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

typedef unsigned long long u64;
typedef unsigned int u32;

// Every per-game routine is __host__ __device__ so that tests/hostcheck can instantiate the very same
// source on the CPU and compare it with the oracle where no GPU exists (test-only; libccx.so has no
// host compute path).
#define CCX_HD __host__ __device__ __forceinline__
#ifdef __CUDA_ARCH__
#define ccx_popc(x) __popc(x)
#define ccx_popcll(x) __popcll(x)
#define ccx_umulhi(a, b) __umulhi((a), (b))
#define ccx_clz(x) __clz(x)
#define ccx_clzll(x) __clzll((long long)(x))
#define ccx_ffs(x) __ffs(x)
#else
#define ccx_popc(x) __builtin_popcount(x)
#define ccx_popcll(x) __builtin_popcountll(x)
#define ccx_umulhi(a, b) ((u32)(((u64)(u32)(a) * (u64)(u32)(b)) >> 32))
#define ccx_clz(x) ((x) ? __builtin_clz(x) : 32)
#define ccx_clzll(x) ((x) ? __builtin_clzll(x) : 64)
#define ccx_ffs(x) __builtin_ffs(x)
#endif

// 7x7 board in a 64-bit word with row stride 8: bit = 8*r + c.  Column 7 and row 7 are guard bits.
#define CCX_VALID 0x007F7F7F7F7F7F7FULL
// board.py:96-111: player 1 wins on diagonals k=4,5,6 -> (0,4)(1,5)(2,6)(0,5)(1,6)(0,6)
#define CCX_TARGET_P1 ((1ULL << 4) | (1ULL << 5) | (1ULL << 6) | (1ULL << 13) | (1ULL << 14) | (1ULL << 22))
// player 2 wins on diagonals -4,-5,-6 -> (4,0)(5,1)(6,2)(5,0)(6,1)(6,0)
#define CCX_TARGET_P2 ((1ULL << 32) | (1ULL << 40) | (1ULL << 41) | (1ULL << 48) | (1ULL << 49) | (1ULL << 50))
// Board() start position (board.py:20-26, 42-46)
#define CCX_START_OCC1 ((1ULL << 48) | (1ULL << 40) | (1ULL << 49) | (1ULL << 32) | (1ULL << 41) | (1ULL << 50))
#define CCX_START_OCC2 ((1ULL << 6) | (1ULL << 14) | (1ULL << 5) | (1ULL << 22) | (1ULL << 13) | (1ULL << 4))
#define CCX_START_CELLS1 (48ULL | (40ULL << 8) | (49ULL << 16) | (32ULL << 24) | (41ULL << 32) | (50ULL << 40))
#define CCX_START_CELLS2 (6ULL | (14ULL << 8) | (5ULL << 16) | (22ULL << 24) | (13ULL << 32) | (4ULL << 40))
#define CCX_START_META 0x00000000FFFFFFFFULL
#define CCX_HIST_EMPTY 0xFFFFFFFFFFFFFFFFULL

// board.py:33-40 direction order: N(-1,0) E(0,+1) SE(+1,+1) S(+1,0) W(0,-1) NW(-1,-1)
template <int D> CCX_HD u64 shd(u64 x)
{
    if (D == 0) return x >> 8;
    if (D == 1) return x << 1;
    if (D == 2) return x << 9;
    if (D == 3) return x << 8;
    if (D == 4) return x >> 1;
    return x >> 9;
}

// One flood-fill round in direction D: all landings of mirror jumps (board.py:172-201) from the
// frontier set F.  `occ` excludes the moving checker (board.py:158), `empty` = ~occ & VALID.
// A jump over a pivot at distance s needs cells 1..s-1 empty, cell s occupied, cells s+1..2s empty.
template <int D> CCX_HD u64 jump_dir(u64 F, u64 occ, u64 empty)
{
    u64 a1 = shd<D>(F);
    u64 L = shd<D>(a1 & occ) & empty;                                   // s = 1
    u64 m1 = a1 & empty;
    u64 a2 = shd<D>(m1);
    L |= shd<D>(shd<D>(a2 & occ) & empty) & empty;                      // s = 2
    u64 m2 = a2 & empty;
    u64 a3 = shd<D>(m2);
    L |= shd<D>(shd<D>(shd<D>(a3 & occ) & empty) & empty) & empty;      // s = 3 (edge to edge on 7x7)
    return L;
}

CCX_HD u64 jump_round(u64 F, u64 occ, u64 empty)
{
    return jump_dir<0>(F, occ, empty) | jump_dir<1>(F, occ, empty) | jump_dir<2>(F, occ, empty) |
           jump_dir<3>(F, occ, empty) | jump_dir<4>(F, occ, empty) | jump_dir<5>(F, occ, empty);
}

CCX_HD u64 neighbours(u64 o)
{
    return shd<0>(o) | shd<1>(o) | shd<2>(o) | shd<3>(o) | shd<4>(o) | shd<5>(o);
}

// Board.get_valid_moves for the side owning `cells` (board.py:215-222).  dest[id] = walks | jump closure.
// Jump parity lemma (SURVEY.md §7.3): jump landings keep (row&1, col&1) of the origin, walk cells do
// not, so the reference's pre-marking of walk cells (board.py:148,155) never prunes a jump chain and
// the legal set is exactly walks ∪ transitive closure.
// The six flood fills run as ONE loop whose body is a single closure round of the thread's current
// checker; a thread that finishes a checker moves on to its next one inside the same loop, so a warp
// iterates max_lanes(sum_checkers rounds) times instead of sum_checkers(max_lanes rounds).
CCX_HD void movegen(u64 occ_all, u64 cells, u64 (&dest)[6])
{
#pragma unroll
    for (int k = 0; k < 6; k++) dest[k] = 0;
    int id = 0;
    u64 o = 1ULL << (cells & 0xFF);
    u64 occ = occ_all & ~o;
    u64 empty = ~occ & CCX_VALID;
    u64 walks = neighbours(o) & empty;
    u64 F = o, reach = 0;
    for (;;) {
        u64 nw = jump_round(F, occ, empty) & ~(reach | o);
        reach |= nw;
        F = nw;
        if (F == 0) {
            u64 d = walks | reach;
#pragma unroll
            for (int k = 0; k < 6; k++) if (id == k) dest[k] = d;
            if (++id == 6) break;
            o = 1ULL << ((cells >> (8 * id)) & 0xFF);
            occ = occ_all & ~o;
            empty = ~occ & CCX_VALID;
            walks = neighbours(o) & empty;
            F = o;
            reach = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Ray formulation of the mirror jumps (board.py:172-201), one source cell at a time.
//
// The six hex directions lie on three line families through a cell: its row (E/W, bit stride 1), its column
// (N/S, stride 8) and its diagonal (SE/NW, stride 9).  For each line the occupancy is gathered into a 7-bit
// index (shift+mask for rows, one multiply for columns/diagonals), a 6,272-byte table answers "where can a
// checker at position `pos` of a line of length `len` with occupancy `o7` land" for BOTH directions at once,
// and the 7-bit answer is scattered back onto the board with one more multiply.  ~65 integer instructions per
// expanded cell instead of ~300 per set-parallel closure round.
#define CCX_JT_BYTES (7 * 7 * 128)

// table entry: landings along a line.  A jump over the first occupied cell b in a direction lands at 2b - pos
// if that cell is on the line and every cell between b and the landing (inclusive) is empty.
CCX_HD uint8_t jump_line_entry(int len, int pos, int o7)
{
    int occ = o7 & ((1 << len) - 1);
    int out = 0;
    for (int dir = -1; dir <= 1; dir += 2) {
        int b = pos + dir;
        while (b >= 0 && b < len && !((occ >> b) & 1)) b += dir;
        if (b < 0 || b >= len) continue;
        int l = 2 * b - pos;
        if (l < 0 || l >= len) continue;
        bool clear = true;
        for (int q = b + dir; q != l + dir; q += dir) if ((occ >> q) & 1) clear = false;
        if (clear) out |= 1 << l;
    }
    return (uint8_t)out;
}

CCX_HD void build_jump_table(uint8_t *T, int first, int step)       // T[(len-1)*896 + pos*128 + o7]
{
    for (int e = first; e < CCX_JT_BYTES; e += step) {
        int len = e / 896 + 1, pos = (e / 128) % 7, o7 = e % 128;
        T[e] = pos < len ? jump_line_entry(len, pos, o7) : 0;
    }
}

// all mirror-jump landings from cell i on occupancy `occ` (mover lifted), not yet masked by visited cells
CCX_HD u64 expand_cell(int i, u64 occ, const uint8_t *__restrict__ T)
{
    const int r = i >> 3, c = i & 7;
    // row: cells (r, 0..6), index along the line = column
    u32 row7 = (u32)(occ >> (8 * r)) & 0x7Fu;
    u64 L = (u64)T[6 * 896 + c * 128 + row7] << (8 * r);
    // column: cells (0..6, c), index = row; gather bits 8j -> j with one multiply (no carries: all partial
    // products land on distinct bits)
    u64 colx = (occ >> c) & 0x0001010101010101ULL;
    u32 col7 = (u32)((colx * 0x0000040810204081ULL) >> 42) & 0x7Fu;
    u64 colr = ((u64)T[6 * 896 + r * 128 + col7] * 0x0002040810204081ULL) & 0x0001010101010101ULL;
    L |= colr << c;
    // diagonal (SE/NW): cells (j, j+k) for k = c - r >= 0, or (j-k, j) for k < 0; bits 9j + shift
    const int k = c - r;
    const int sh = k >= 0 ? k : -8 * k;
    const int len = 7 - (k >= 0 ? k : -k);
    const int pos = k >= 0 ? r : c;
    u64 diax = (occ >> sh) & 0x0040201008040201ULL;
    u32 dia7 = (u32)((diax * 0x0001010101010101ULL) >> 48) & 0x7Fu;
    u64 diar = ((u64)T[(len - 1) * 896 + pos * 128 + dia7] * 0x0001010101010101ULL) & 0x0040201008040201ULL;
    L |= diar << sh;
    return L;
}

// Second table layout ("occupancy-major"): T2[(len-1)*1024 + o7*8 + pos].  Lines of a sparse board share a handful of occupancy
// patterns, so lanes of a warp mostly differ in `pos`: with the pattern-major layout above those lanes hit DIFFERENT words of
// the SAME bank (bank = (o7 >> 2) & 31 whatever pos is), here they hit the same 8-byte row (a broadcast).
#define CCX_JT2_BYTES (7 * 128 * 8)

CCX_HD void build_jump_table2(uint8_t *T2, int first, int step)
{
    for (int e = first; e < CCX_JT2_BYTES; e += step) {
        int len = e / 1024 + 1, o7 = (e / 8) % 128, pos = e % 8;
        T2[e] = pos < len ? jump_line_entry(len, pos, o7) : 0;
    }
}

CCX_HD u32 cell_diag_info2(int i)
{
    const int r = i >> 3, c = i & 7, k = c - r;
    const int sh = k >= 0 ? k : -8 * k;
    const int len = 7 - (k >= 0 ? k : -k);
    const int pos = k >= 0 ? r : c;
    return (u32)(sh & 0xFF) | ((u32)(((len > 0 ? len : 1) - 1) * 1024 + (pos & 7)) << 8);
}

CCX_HD u64 expand_cell_lut2(int i, u64 occ, const uint8_t *__restrict__ T2, const u32 *__restrict__ CI2)
{
    const u32 ci = CI2[i];
    const int r = i >> 3, c = i & 7;
    u32 row7 = (u32)(occ >> (8 * r)) & 0x7Fu;
    u64 L = (u64)T2[6 * 1024 + row7 * 8 + c] << (8 * r);
    u64 colx = (occ >> c) & 0x0001010101010101ULL;
    u32 col7 = (u32)((colx * 0x0000040810204081ULL) >> 42) & 0x7Fu;
    u64 colr = ((u64)T2[6 * 1024 + col7 * 8 + r] * 0x0002040810204081ULL) & 0x0001010101010101ULL;
    L |= colr << c;
    const int sh = (int)(ci & 0xFFu);
    u64 diax = (occ >> sh) & 0x0040201008040201ULL;
    u32 dia7 = (u32)((diax * 0x0001010101010101ULL) >> 48) & 0x7Fu;
    u64 diar = ((u64)T2[(ci >> 8) + dia7 * 8] * 0x0001010101010101ULL) & 0x0040201008040201ULL;
    L |= diar << sh;
    return L;
}

// ---------------------------------------------------------------------------------------------------------
// Three-layout formulation (k_step_random_pick, k_step_random_wq, k_play_greedy_tri).  The expensive parts of expand_cell are the two multiplies that GATHER a
// column's / diagonal's occupancy into 7 bits and the two that SCATTER the 7-bit answer back.  Both disappear when the
// occupancy is also kept column-major and diagonal-major (a move flips two bits in each copy) with every line in a BYTE of
// its own — gathering a line is then ONE byte-permute instruction (PRMT picks byte 0-7 of a register pair; bit 7 of every
// byte is a guard bit, so the sign-replicating selector 0x8880 | byte zero-extends it) — and when the column / diagonal
// tables hold 64-bit answers that are already spread over the board (scatter = one shift).
//   T layout: bit 8*c + r            (column c = byte c, index along the line = row)
//   D layout: the nine diagonals k = c - r that are long enough to jump on (|k| <= 4): k = -3..3 in bytes 1..7, the two
//             3-cell diagonals share byte 0 (k = -4 in bits 0-2, k = +4 in bits 4-6); position along the diagonal = r if
//             k >= 0 else c.  Cells of the four corner diagonals (|k| >= 5, no jump possible) map to the dump bit 3.
// Table blob (CCX_JT3_BYTES): row answers u8 [o7][64 cells]; column answers u64 [o7][8 rows], bit 8*l = landing row l in
// column 0; diagonal answers u64 [o7][29], bit 9*l = landing l on the main diagonal, column lp = 0-2: k = -4, 3-5: k = +4
// (occupancy in bits 4-6), 6-9: 4 cells, 10-14: 5, 15-20: 6, 21-27: 7, 28: zeros (corner diagonals).
#define CCX_JT3_ROW 0
#define CCX_JT3_COL (128 * 64)
#define CCX_JT3_DIA (CCX_JT3_COL + 128 * 8 * 8)
#define CCX_JT3_NLP 29
#define CCX_JT3_BYTES (CCX_JT3_DIA + 128 * CCX_JT3_NLP * 8)

CCX_HD int tri_tbit(int cell) { return ((cell & 7) << 3) | (cell >> 3); }
CCX_HD int tri_dbyte(int k) { return (k == -4 || k == 4) ? 0 : k + 4; }
CCX_HD int tri_dbit(int cell)
{
    const int r = cell >> 3, c = cell & 7, k = c - r;
    if (k < -4 || k > 4) return 3;
    return 8 * tri_dbyte(k) + (k == 4 ? 4 : 0) + (k >= 0 ? r : c);
}
CCX_HD int tri_lp(int k, int pos)
{
    const int len = 7 - (k >= 0 ? k : -k);
    if (len < 3) return 28;
    if (len == 3) return (k > 0 ? 3 : 0) + pos;
    return (len == 4 ? 6 : len == 5 ? 10 : len == 6 ? 15 : 21) + pos;
}
// per-cell constants, two words.  lo: diagonal byte selector (0x8880 | byte) | board shift of the diagonal << 16 | byte offset of its
// answer column << 24;  hi: row byte selector (0x8880 | r) | column byte selector (0x8880 | c) << 16
CCX_HD u64 tri_cell_info(int cell)
{
    const int r = cell >> 3, c = cell & 7, k = c - r;
    const int sh = k >= 0 ? k : -8 * k;
    const int sel = (k < -4 || k > 4) ? 4 : tri_dbyte(k);
    const u32 lo = (0x8880u | (u32)sel) | ((u32)(sh & 0xFF) << 16) | ((u32)(tri_lp(k, k >= 0 ? r : c) * 8) << 24);
    const u32 hi = (0x8880u | (u32)r) | ((0x8880u | (u32)c) << 16);
    return (u64)lo | ((u64)hi << 32);
}

CCX_HD void build_jump_table3(uint8_t *T3, int first, int step)
{
    for (int e = first; e < 128 * 64; e += step) {                      // rows: [o7][cell]
        int o7 = e / 64, cell = e % 64;
        T3[CCX_JT3_ROW + e] = ((CCX_VALID >> cell) & 1) ? jump_line_entry(7, cell & 7, o7) : 0;
    }
    u64 *C = reinterpret_cast<u64 *>(T3 + CCX_JT3_COL);
    for (int e = first; e < 128 * 8; e += step) {                       // columns: [o7][row]
        int o7 = e / 8, pos = e % 8;
        u32 m = pos < 7 ? jump_line_entry(7, pos, o7) : 0;
        u64 out = 0;
        for (int l = 0; l < 7; l++) if ((m >> l) & 1) out |= 1ULL << (8 * l);
        C[e] = out;
    }
    u64 *D = reinterpret_cast<u64 *>(T3 + CCX_JT3_DIA);
    for (int e = first; e < 128 * CCX_JT3_NLP; e += step) {             // diagonals: [o7][lp]
        int o7 = e / CCX_JT3_NLP, lp = e % CCX_JT3_NLP;
        int len, pos, occ = o7;
        if (lp < 3) { len = 3; pos = lp; }
        else if (lp < 6) { len = 3; pos = lp - 3; occ = o7 >> 4; }
        else if (lp < 10) { len = 4; pos = lp - 6; }
        else if (lp < 15) { len = 5; pos = lp - 10; }
        else if (lp < 21) { len = 6; pos = lp - 15; }
        else if (lp < 28) { len = 7; pos = lp - 21; }
        else { len = 0; pos = 0; }
        u32 m = len ? jump_line_entry(len, pos, occ) : 0;
        u64 out = 0;
        for (int l = 0; l < 7; l++) if ((m >> l) & 1) out |= 1ULL << (9 * l);
        D[e] = out;
    }
}

#ifdef __CUDA_ARCH__
// PRMT in its default mode (selector nibble = source byte 0-7 | 8 to replicate that byte's sign bit).  __byte_perm() masks the
// selector with 0x7777, which would fill bytes 1-3 with copies instead of zeros, hence the inline PTX.
static __device__ __forceinline__ u32 ccx_byte_of(u32 lo, u32 hi, u32 sel)
{
    u32 d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(lo), "r"(hi), "r"(sel));
    return d;
}
// index of the top set bit of a 32-bit word, -1 for zero (FLO)
static __device__ __forceinline__ int ccx_flo(u32 x)
{
    int d;
    asm("bfind.u32 %0, %1;" : "=r"(d) : "r"(x));
    return d;
}
#else
static inline u32 ccx_byte_of(u32 lo, u32 hi, u32 sel)        // host model of PRMT in its default mode
{
    const u64 v = (u64)lo | ((u64)hi << 32);
    u32 d = 0;
    for (int q = 0; q < 4; q++) {
        const u32 n = (sel >> (4 * q)) & 0xFu, b = (u32)(v >> (8 * (n & 7u))) & 0xFFu;
        d |= (n & 8u ? (b & 0x80u ? 0xFFu : 0u) : b) << (8 * q);
    }
    return d;
}
static inline int ccx_flo(u32 x) { return x ? 31 - __builtin_clz(x) : -1; }
#endif

// all mirror-jump landings from cell i; occ / occT / occD = the occupancy without the mover in the three layouts
CCX_HD u64 expand_cell_tri(int i, u64 occ, u64 occT, u64 occD, const uint8_t *__restrict__ T3, const u64 *__restrict__ CI3)
{
    const u64 ci = CI3[i];
    const u32 clo = (u32)ci, chi = (u32)(ci >> 32);
    const int r8 = i & 0x38;
    const u32 row7 = ccx_byte_of((u32)occ, (u32)(occ >> 32), chi);
    u64 L = (u64)T3[CCX_JT3_ROW + row7 * 64 + i] << r8;
    const u32 col7 = ccx_byte_of((u32)occT, (u32)(occT >> 32), chi >> 16);
    L |= *reinterpret_cast<const u64 *>(T3 + CCX_JT3_COL + col7 * 64 + r8) << (i & 7);
    const u32 dia7 = ccx_byte_of((u32)occD, (u32)(occD >> 32), clo);
    L |= *reinterpret_cast<const u64 *>(T3 + CCX_JT3_DIA + dia7 * (CCX_JT3_NLP * 8) + (clo >> 24)) << ((clo >> 16) & 0xFFu);
    return L;
}

// Board.get_valid_moves (board.py:215-222) with the ray formulation.  Same single-loop structure as movegen():
// the loop body expands ONE cell of the thread's current checker (origin first, then every newly reached
// landing cell), and a thread that exhausts a checker moves on to its next one inside the same loop.
CCX_HD void movegen_rays(u64 occ_all, u64 cells, u64 (&dest)[6], const uint8_t *__restrict__ T)
{
#pragma unroll
    for (int k = 0; k < 6; k++) dest[k] = 0;
    int id = 0;
    u64 o = 1ULL << (cells & 0xFF);
    u64 occ = occ_all & ~o;
    u64 todo = o, reach = 0;
    for (;;) {
        // any expansion order gives the same closure; the top set bit is the cheapest to find on the GPU (one FLO)
#ifdef __CUDA_ARCH__
        int i = 63 - __clzll((long long)todo);
#else
        int i = 63 - __builtin_clzll(todo);
#endif
        todo ^= 1ULL << i;
        u64 nw = expand_cell(i, occ, T) & ~(reach | o);
        reach |= nw;
        todo |= nw;
        if (todo == 0) {
            u64 d = (neighbours(o) & ~occ & CCX_VALID) | reach;
#pragma unroll
            for (int k = 0; k < 6; k++) if (id == k) dest[k] = d;
            if (++id == 6) break;
            o = 1ULL << ((cells >> (8 * id)) & 0xFF);
            occ = occ_all & ~o;
            todo = o;
            reach = 0;
        }
    }
}

// k-th (0-based) set bit of m, ascending; requires k < popc(m)
CCX_HD int select64(u64 m, u32 k)
{
    u32 lo = (u32)m, hi = (u32)(m >> 32);
    u32 c = ccx_popc(lo);
    u32 w = lo; int base = 0;
    if (k >= c) { w = hi; base = 32; k -= c; }
    c = ccx_popc(w & 0xFFFFu); if (k >= c) { w >>= 16; base += 16; k -= c; }
    c = ccx_popc(w & 0xFFu);   if (k >= c) { w >>= 8;  base += 8;  k -= c; }
    c = ccx_popc(w & 0xFu);    if (k >= c) { w >>= 4;  base += 4;  k -= c; }
    c = ccx_popc(w & 0x3u);    if (k >= c) { w >>= 2;  base += 2;  k -= c; }
    c = w & 1u;              if (k >= c) { base += 1; }
    return base;
}

CCX_HD int check_win(u64 occ1, u64 occ2)      // board.py:89-111
{
    if ((occ1 & CCX_TARGET_P1) == CCX_TARGET_P1) return 1;
    if ((occ2 & CCX_TARGET_P2) == CCX_TARGET_P2) return 2;
    return 0;
}

// Philox4x32-10 (Salmon et al., SC'11); key = seed, counter = (c0, c1, game id lo, game id hi)
struct Philox4 { u32 x, y, z, w; };
CCX_HD Philox4 philox4x32_10(u32 k0, u32 k1, u32 c0, u32 c1, u32 c2, u32 c3)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        u32 h0 = ccx_umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        u32 h1 = ccx_umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        u32 n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    Philox4 o = {c0, c1, c2, c3};
    return o;
}

// The per-game record the env kernels keep in registers, from the side to move's point of view.
struct Game {
    u64 occ_me, occ_op, cells_me, cells_op, meta;
};

// Board.place for checker `id` of the side to move (board.py:226-250): occupancy swap, id->cell
// rewrite in place (:235-238), last-two-moves shift (:246-248), ply++, side flip.
CCX_HD void apply_move(Game &g, int id, int from, int to)
{
    g.occ_me ^= (1ULL << from) | (1ULL << to);
    g.cells_me = (g.cells_me & ~(0xFFULL << (8 * id))) | ((u64)to << (8 * id));
    u64 meta = g.meta;
    u64 ply = ((meta >> 32) + 1) & 0xFFFF;
    g.meta = (meta & 0xFFFF000000000000ULL) ^ (1ULL << 48) | (ply << 32) | ((meta & 0xFFFF) << 16) |
             (u64)from | ((u64)to << 8);
    u64 t;
    t = g.occ_me; g.occ_me = g.occ_op; g.occ_op = t;
    t = g.cells_me; g.cells_me = g.cells_op; g.cells_op = t;
}

CCX_HD void push_hist(u64 &lo, u64 &hi, int to)     // board.py:246-248 (destinations only)
{
    hi = (hi << 8) | (lo >> 56);
    lo = (lo << 8) | (u64)to;
}

CCX_HD int level_of(int cell) { return (cell >> 3) - (cell & 7) + 6; }   // board_utils.py:3-7: human row - 1

CCX_HD int winner_of(const Game &g)     // check_win in absolute player numbering
{
    bool p2 = (g.meta >> 48) & 1;
    return check_win(p2 ? g.occ_op : g.occ_me, p2 ? g.occ_me : g.occ_op);
}

CCX_HD void reset_start(Game &g)
{
    g.occ_me = CCX_START_OCC1; g.occ_op = CCX_START_OCC2;
    g.cells_me = CCX_START_CELLS1; g.cells_op = CCX_START_CELLS2;
    g.meta = CCX_START_META;
}

// selfplay.make_random_move's choice (selfplay.py:93-98) from two 32-bit random words; returns the
// checker id, fills from/to.  Requires at least one non-empty mask.
CCX_HD int pick_random(const Game &g, const u64 (&dest)[6], u32 nonempty, u32 r0, u32 r1, int &from, int &to)
{
    int j = (int)ccx_umulhi(r0, nonempty);
    int id = 0, rank = 0; u64 m = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) {         // j-th checker (id order) that can move
        bool ne = dest[k] != 0;
        if (ne && rank == j) { id = k; m = dest[k]; }
        rank += ne;
    }
    to = select64(m, ccx_umulhi(r1, (u32)ccx_popcll(m)));
    from = (int)((g.cells_me >> (8 * id)) & 0xFF);
    return id;
}

// ---------------------------------------------------------------------------------------------------------
// Three-layout move generation and the pick-first random ply.  The kernels pass tables staged in shared memory, the host
// tests the same tables built on the CPU.
struct TriTables {
    const uint8_t *sT; const u64 *sNB, *sCI, *sO, *sOT, *sOD;     // build_jump_table3, [64] on-board neighbours, tri_cell_info, 1 << cell, 1 << tri_tbit, 1 << tri_dbit
    const u32 *sSel;                                              // [128] sel7_entry, staged by the kernels that use select64_step
    const u64 *sW;                                                // build_jump_table_wide, staged by the one-wave carry kernel instead of sT / sCI
};

// occupancy in the T and D layouts from the twelve checker cells
CCX_HD void tri_build(u64 cells_a, u64 cells_b, const u64 *__restrict__ sOT, const u64 *__restrict__ sOD, u64 &occT, u64 &occD)
{
    occT = 0; occD = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        int a = (int)((cells_a >> (8 * k)) & 0x3F), b = (int)((cells_b >> (8 * k)) & 0x3F);
        occT |= sOT[a] | sOT[b];
        occD |= sOD[a] | sOD[b];
    }
}

// Board.get_valid_moves (board.py:215-222) with the three-layout expansion; same single-loop structure as movegen_rays.
// WIDE: over the wide tables (T.sW), for the kernel that stages them instead of T.sT / T.sCI.
CCX_HD u64 expand_cell_carry(int c, u64 occ, u64 occT, u64 occD, const u64 *__restrict__ W);     // below, with the wide tables
template <bool WIDE = false>
CCX_HD void movegen_tri(u64 occ_all, u64 occT_all, u64 occD_all, u64 cells, u64 (&dest)[6], const TriTables &T)
{
#pragma unroll
    for (int k = 0; k < 6; k++) dest[k] = 0;
    int id = 0, cell = (int)(cells & 0x3F);
    u64 o = T.sO[cell], occ = occ_all & ~o, occT = occT_all & ~T.sOT[cell], occD = occD_all & ~T.sOD[cell];
    u64 todo = o, reach = 0;
    for (;;) {
        int c = 63 - ccx_clzll(todo);
        todo ^= T.sO[c];
        u64 nw = (WIDE ? expand_cell_carry(c, occ, occT, occD, T.sW) : expand_cell_tri(c, occ, occT, occD, T.sT, T.sCI)) & ~(reach | o);
        reach |= nw;
        todo |= nw;
        if (todo == 0) {
            u64 d = (T.sNB[cell] & ~occ) | reach;
#pragma unroll
            for (int k = 0; k < 6; k++) if (id == k) dest[k] = d;
            if (++id == 6) break;
            cell = (int)((cells >> (8 * id)) & 0x3F);
            o = T.sO[cell]; occ = occ_all & ~o; occT = occT_all & ~T.sOT[cell]; occD = occD_all & ~T.sOD[cell];
            todo = o; reach = 0;
        }
    }
}

// One checker's jump flood fill: the mover's bit, the occupancy without it in the three layouts, the cells still to expand
// and the landings reached so far.
struct JumpFill {
    u64 o, occ, occT, occD, todo, reach;
};

CCX_HD JumpFill fill_start(int cell, u64 occ_all, u64 occT_all, u64 occD_all, const TriTables &T)
{
    JumpFill f;
    f.o = 1ULL << cell;            // a shift, not sO[cell]: one shared-memory load fewer (that pipe bounded the work-queue kernel)
    f.occ = occ_all & ~f.o; f.occT = occT_all & ~T.sOT[cell]; f.occD = occD_all & ~T.sOD[cell];
    f.todo = f.o; f.reach = 0;
    return f;
}

// expand one cell of the fill (any order gives the same closure; the top set bit is the cheapest to find on the GPU)
CCX_HD void fill_step(JumpFill &f, const TriTables &T)
{
    const int c = 63 - ccx_clzll(f.todo);
    f.todo ^= 1ULL << c;
    const u64 nw = expand_cell_tri(c, f.occ, f.occT, f.occD, T.sT, T.sCI) & ~(f.reach | f.o);
    f.reach |= nw;
    f.todo |= nw;
}

// Bit k set iff checker k of the side to move has an empty neighbour (a walk).  The neighbour relation is symmetric, so the
// checkers with a walk are the mover's cells among the neighbours of the empty cells: one set-parallel pass for all six.
CCX_HD u32 walk_movable(u64 occ_me, u64 occ_all, u64 cells_me)
{
    const u64 w = occ_me & neighbours(~occ_all & CCX_VALID);
    u32 b = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) b |= (u32)((w >> ((cells_me >> (8 * k)) & 0x3F)) & 1) << k;
    return b;
}

// pick_random's choice made before any destination set is known.  pick_random only needs WHICH checkers can move and the
// full set of the one it picks.  A checker can move iff it has a walk or its first jump lands (a jump closure is empty iff
// its first expansion is), so only the rare checker without an empty neighbour costs an expansion here, and only the picked
// checker's closure is flood-filled.  Same Philox words, same arithmetic and id order, hence the same move as
// pick_random over movegen's six sets.
// pick_first_start picks the checker with r0 and starts its fill: returns the checker id and sets from / f, or -1 when no
// checker can move.  Once the fill is done (f.todo == 0), pick_first_to draws the destination with r1.
CCX_HD int pick_first_start(const Game &g, u64 occT_all, u64 occD_all, u32 r0, const TriTables &T, int &from, JumpFill &f)
{
    const u64 occ_all = g.occ_me | g.occ_op;
    u32 movable = walk_movable(g.occ_me, occ_all, g.cells_me);
    u32 nowalk = ~movable & 0x3Fu;
    while (nowalk) {                          // ~0.008 checkers per game-ply in random play
        const int k = ccx_ffs(nowalk) - 1;
        nowalk &= nowalk - 1;
        JumpFill p = fill_start((int)((g.cells_me >> (8 * k)) & 0x3F), occ_all, occT_all, occD_all, T);
        fill_step(p, T);
        if (p.reach) movable |= 1u << k;
    }
    if (!movable) return -1;
    const int id = select64(movable, ccx_umulhi(r0, (u32)ccx_popc(movable)));
    from = (int)((g.cells_me >> (8 * id)) & 0x3F);
    f = fill_start(from, occ_all, occT_all, occD_all, T);
    return id;
}

CCX_HD int pick_first_to(u64 occ_all, int from, const JumpFill &f, u32 r1, const TriTables &T)
{
    const u64 m = (T.sNB[from] & ~occ_all) | f.reach;
    return select64(m, ccx_umulhi(r1, (u32)ccx_popcll(m)));
}

// the whole ply in one call: returns the checker id and sets from / to, or -1 when no checker can move
CCX_HD int pick_random_first(const Game &g, u64 occT_all, u64 occD_all, u32 r0, u32 r1, const TriTables &T, int &from, int &to)
{
    JumpFill f;
    const int id = pick_first_start(g, occT_all, occD_all, r0, T, from, f);
    if (id < 0) return -1;
    while (f.todo) fill_step(f, T);
    to = pick_first_to(g.occ_me | g.occ_op, from, f, r1, T);
    return id;
}

// ---------------------------------------------------------------------------------------------------------
// The ply of k_step_random_carry: the same choice as pick_first_start / pick_first_to, with shorter dependent chains.

// Rank table of the step path's selects (CCX_SEL7_BYTES): entry v of 128 holds the positions of v's set bits in ascending
// order, 3 bits each, so the r-th set bit of a 7-bit value is (entry >> 3r) & 7.
#define CCX_SEL7_BYTES (128 * 4)
CCX_HD u32 sel7_entry(u32 v)
{
    u32 e = 0, n = 0;
    for (u32 b = 0; b < 7; b++)
        if ((v >> b) & 1u) e |= b << (3 * n++);
    return e;
}

// the r-th (0-based) set bit of a 7-bit value v; requires r < popc(v)
CCX_HD u32 sel7_rank(const u32 *__restrict__ sSel, u32 v, u32 r) { return (sSel[v] >> (3 * r)) & 7u; }

// select64(m, k) with two popcount levels instead of six: the 32-bit half, then the byte from three prefix popcounts of the
// half taken in parallel, then the bit from the rank table (bit 7 of the byte, which the table does not cover, by a compare).
CCX_HD int select64_step(u64 m, u32 k, const u32 *__restrict__ sSel)
{
    const u32 lo = (u32)m, hi = (u32)(m >> 32), c = ccx_popc(lo);
    const bool up = k >= c;
    const u32 w = up ? hi : lo;
    k -= up ? c : 0u;
    const u32 c1 = ccx_popc(w & 0xFFu), c2 = ccx_popc(w & 0xFFFFu), c3 = ccx_popc(w & 0xFFFFFFu);
    const bool p1 = k >= c1, p2 = k >= c2, p3 = k >= c3;        // p3 implies p2 implies p1
    const u32 below = p2 ? (p3 ? c3 : c2) : (p1 ? c1 : 0u);
    const u32 sh = p2 ? (p3 ? 24u : 16u) : (p1 ? 8u : 0u);
    const u32 v = (w >> sh) & 0xFFu, r = k - below;
    const u32 pos = r < (u32)ccx_popc(v & 0x7Fu) ? sel7_rank(sSel, v & 0x7Fu, r) : 7u;
    return (int)((up ? 32u : 0u) + sh + pos);
}

// The cells of the mover's checkers without an empty neighbour: occ_me & ~neighbours(empty), with the six shifts of
// neighbours() paired into four, (e | e << 1) << 8 | e << 1 | (e | e >> 1) >> 8 | e >> 1.  Bits shifted onto the guard
// column and row are not the mover's, so no mask is needed.
CCX_HD u64 nowalk_cells(u64 occ_me, u64 occ_all)
{
    const u64 e = ~occ_all & CCX_VALID, l = e << 1, r = e >> 1;
    return occ_me & ~(((e | l) << 8) | l | ((e | r) >> 8) | r);
}

// tri_cell_info's constants computed from the cell with ALU instructions, for the carry kernel's fill: with them the three
// table loads of an expansion depend on c through a few ALU instructions instead of one more shared-memory load.  With
// k = col - r, the diagonal's PRMT selectors are sums with 0x8894 - 4 = 0x8890, so nibbles 1-3 stay 8 or 9 (the sign of a byte
// whose bit 7 is a guard bit: zero) and nibble 0 is the byte:
//   dsel: the diagonal's byte in the D layout, k + 4 for k = -4..3 and 0 for k = 4 (`& ((x - 1) | 7)` clears the 8 of
//         k + 4 = 8 and nothing else); for the corner diagonals |k| >= 5 a nibble >= 8, a zero byte (o7 = 0: no landing);
//   lp8: byte offset of the answer column, 8 * (first column of the line + position along it), position = min(r, col) (r if
//        k >= 0 else col); the first column is byte 4 - k of CCX_DBASE (k = 4..-3), and k = -4 and the corners select a sign (0).
//   sh:  the board shift of the diagonal, k if k >= 0 else -8k.
#define CCX_DBASE_LO 0x78503018u                 // 8 * {3, 6, 10, 15} for k = 4, 3, 2, 1
#define CCX_DBASE_HI 0x305078A8u                 // 8 * {21, 15, 10, 6} for k = 0, -1, -2, -3
struct CarryCell { u32 rsel, csel, dsel, lp8, sh; };
CCX_HD CarryCell carry_cell(int c)
{
    const int r = c >> 3, col = c & 7, k = col - r;
    const u32 x = (u32)k + 0x8894u;
    const u32 base8 = ccx_byte_of(CCX_DBASE_LO, CCX_DBASE_HI, 0x8894u - (u32)k);
    CarryCell q;
    q.rsel = 0x8880u + (u32)r;                // r, col < 8: an add, not an OR
    q.csel = 0x8880u + (u32)col;
    q.dsel = x & ((x - 1u) | 7u);
    q.lp8 = base8 + 8u * (u32)(r < col ? r : col);
    q.sh = (u32)(k > -8 * k ? k : -8 * k);
    return q;
}

// expand_cell_tri with carry_cell's constants
CCX_HD u64 expand_cell_carry(int c, u64 occ, u64 occT, u64 occD, const uint8_t *__restrict__ T3)
{
    CarryCell q = carry_cell(c);
    const int r8 = c & 0x38;
    const u32 row7 = ccx_byte_of((u32)occ, (u32)(occ >> 32), q.rsel);
    u64 L = (u64)T3[CCX_JT3_ROW + row7 * 64 + c] << r8;
    const u32 col7 = ccx_byte_of((u32)occT, (u32)(occT >> 32), q.csel);
    L |= *reinterpret_cast<const u64 *>(T3 + CCX_JT3_COL + col7 * 64 + r8) << (c & 7);
    const u32 dia7 = ccx_byte_of((u32)occD, (u32)(occD >> 32), q.dsel);
#ifdef __CUDA_ARCH__
    asm("" : "+r"(q.lp8));   // lp8 is ready before dia7: one IMAD after the PRMT, not (dia7 * 29 + pos) * 8 + base8
#endif
    L |= *reinterpret_cast<const u64 *>(T3 + CCX_JT3_DIA + dia7 * (CCX_JT3_NLP * 8) + q.lp8) << q.sh;
    return L;
}

// Wide answer tables (CCX_JTW_BYTES, u64 [3][o7][cell]): build_jump_table3's row, column and diagonal answers for every cell,
// each already shifted to its place on the board, so an expansion is three PRMTs, three o7 * 512 + 8c addresses and three
// 8-byte loads, with no shift of an answer and no per-cell column offset or board shift.  Cells off the board and the
// corner diagonals' cells (whose selector picks a zero byte) hold 0.
#define CCX_JTW_ROW 0
#define CCX_JTW_COL (128 * 64)
#define CCX_JTW_DIA (2 * 128 * 64)
#define CCX_JTW_BYTES (3 * 128 * 64 * 8)
CCX_HD void build_jump_table_wide(u64 *W, const uint8_t *T3, int first, int step)
{
    for (int e = first; e < 128 * 64; e += step) {
        const int o7 = e / 64, c = e % 64, r = c >> 3, col = c & 7, k = col - r;
        const bool on = (CCX_VALID >> c) & 1, dia = on && k >= -4 && k <= 4;
        const u64 ci = tri_cell_info(c);
        W[CCX_JTW_ROW + e] = on ? (u64)T3[CCX_JT3_ROW + o7 * 64 + c] << (c & 0x38) : 0;
        W[CCX_JTW_COL + e] = on ? *reinterpret_cast<const u64 *>(T3 + CCX_JT3_COL + o7 * 64 + 8 * r) << col : 0;
        W[CCX_JTW_DIA + e] = dia ? *reinterpret_cast<const u64 *>(T3 + CCX_JT3_DIA + o7 * (CCX_JT3_NLP * 8) + ((u32)ci >> 24))
                                       << ((ci >> 16) & 0xFF) : 0;
    }
}

// expand_cell_carry over the wide tables (of carry_cell only the selectors)
CCX_HD u64 expand_cell_carry(int c, u64 occ, u64 occT, u64 occD, const u64 *__restrict__ W)
{
    const CarryCell q = carry_cell(c);
    const u32 row7 = ccx_byte_of((u32)occ, (u32)(occ >> 32), q.rsel);
    const u32 col7 = ccx_byte_of((u32)occT, (u32)(occT >> 32), q.csel);
    const u32 dia7 = ccx_byte_of((u32)occD, (u32)(occD >> 32), q.dsel);
#ifdef __CUDA_ARCH__
    // W is in shared memory.  One IMAD per address, o7 * 512 + (base + 8c), with the table's offset in the load: written
    // with plain indexing, ptxas forms (o7 * 64 + c) * 8 and adds the base per load.
    const u32 wc = (u32)__cvta_generic_to_shared(W) + 8u * (u32)c;
    u64 a, b, d;
    asm("ld.shared.u64 %0, [%1];" : "=l"(a) : "r"(wc + row7 * 512u));
    asm("ld.shared.u64 %0, [%1+65536];" : "=l"(b) : "r"(wc + col7 * 512u));
    asm("ld.shared.u64 %0, [%1+131072];" : "=l"(d) : "r"(wc + dia7 * 512u));
    return a | b | d;
#else
    return W[CCX_JTW_ROW + row7 * 64 + c] | W[CCX_JTW_COL + col7 * 64 + c] | W[CCX_JTW_DIA + dia7 * 64 + c];
#endif
}

// a | b for words without a common set bit: an add per 32-bit half, which no carry leaves.  ptxas may issue an add to the
// IMAD pipe (IMAD.IADD, VIADD); an OR goes to the ALU pipe, which the carry kernel's integer work loads most.
CCX_HD u64 or_disjoint(u64 a, u64 b)
{
    u32 lo = (u32)a + (u32)b, hi = (u32)(a >> 32) + (u32)(b >> 32);
#ifdef __CUDA_ARCH__
    asm("" : "+r"(lo), "+r"(hi));            // else the halves are fused back into a 64-bit add with a carry
#endif
    return (u64)lo | ((u64)hi << 32);
}

// the answer tables the carry kernel expands on: the wide ones (WIDE) or build_jump_table3's
template <bool WIDE>
CCX_HD auto carry_tables(const TriTables &T)
{
    if constexpr (WIDE) return T.sW; else return T.sT;
}

// fill_step for k_step_random_carry: the same cell order (the top set bit, from two independent FLOs: the high word's index
// | 32 is -1 when that word is empty, so a signed max picks the right one) and expand_cell_carry on either table set
template <class TAB>
CCX_HD void fill_step_carry(JumpFill &f, const TAB *__restrict__ tab)
{
    const int h = ccx_flo((u32)(f.todo >> 32)) | 32, l = ccx_flo((u32)f.todo);
    const int c = h > l ? h : l;
    f.todo ^= 1ULL << c;
    const u64 nw = expand_cell_carry(c, f.occ, f.occT, f.occD, tab) & ~(f.reach | f.o);
    f.reach = or_disjoint(f.reach, nw);
    f.todo |= nw;
}

// The fill of the checker on cell `from`, seeded with its walks and with its first step taken: the expansion of the origin.  A
// line's answer does not depend on the occupancy of the cell it is asked for (jump_line_entry never reads bit `pos`), so the
// origin expands on the full occupancy: its three loads need neither FLO nor the mover-free words and issue alongside
// sOT / sOD / sNB[from].  Its landings are empty cells other than the origin and, by the parity lemma above movegen, not walks,
// so nothing is masked.  No jump lands on a walk cell either, so the seed prunes nothing, and when the fill is done f.reach
// is the whole destination set.  f.todo may be 0 on return (28.8 % of plies in random play).
template <bool WIDE = false>
CCX_HD JumpFill carry_fill_start(int from, u64 occ_all, u64 occT_all, u64 occD_all, const TriTables &T)
{
    JumpFill f;
    f.o = 1ULL << from;
    f.occ = occ_all & ~f.o; f.occT = occT_all & ~T.sOT[from]; f.occD = occD_all & ~T.sOD[from];
    f.todo = expand_cell_carry(from, occ_all, occT_all, occD_all, carry_tables<WIDE>(T));
    f.reach = (T.sNB[from] & ~occ_all) | f.todo;
    return f;
}

// pick_first_start for k_step_random_carry, with the same choice; the fill starts with carry_fill_start.  The pick is made
// speculatively for the common case in which every checker has a walk (all but ~0.8 % of plies in random play): then all six
// can move, popc = 6 and the rank table maps j to j, so the checker is umulhi(r0, 6) and the fill's loads issue alongside the
// test instead of after the walk bits, the popcount and the rank lookup.  Otherwise the speculative start is dropped and the
// checker is picked by the rank table over the exact movable set; a checker without a walk can move iff its origin's
// expansion lands (on the full occupancy, as above).  The fallback's work stays behind its branch: it starts from the
// no-walk cells, which the test computes anyway.
template <bool WIDE = false>
CCX_HD int carry_ply_start(const Game &g, u64 occT_all, u64 occD_all, u32 r0, const TriTables &T, int &from, JumpFill &f)
{
    const u64 occ_all = g.occ_me | g.occ_op;
    int id = (int)ccx_umulhi(r0, 6u);
    from = (int)ccx_byte_of((u32)g.cells_me, (u32)(g.cells_me >> 32), 0x8880u + (u32)id);
    f = carry_fill_start<WIDE>(from, occ_all, occT_all, occD_all, T);
    u64 nowalk = nowalk_cells(g.occ_me, occ_all);
    if (!nowalk) return id;
    u64 stuck = 0;                            // checkers that cannot move at all
    do {                                      // ~0.008 checkers per game-ply in random play
        const int c = 63 - ccx_clzll(nowalk);
        nowalk ^= 1ULL << c;
        if (!expand_cell_carry(c, occ_all, occT_all, occD_all, carry_tables<WIDE>(T))) stuck |= 1ULL << c;
    } while (nowalk);
    u64 cells = g.cells_me;
#ifdef __CUDA_ARCH__
    asm volatile("" : "+l"(cells));           // else the six extracts below are hoisted onto the common path
#endif
    u32 movable = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) movable |= (u32)(~stuck >> ((cells >> (8 * k)) & 0x3F) & 1) << k;
    if (!movable) return -1;
    id = (int)sel7_rank(T.sSel, movable, ccx_umulhi(r0, (u32)ccx_popc(movable)));
    from = (int)ccx_byte_of((u32)g.cells_me, (u32)(g.cells_me >> 32), 0x8880u + (u32)id);
    f = carry_fill_start<WIDE>(from, occ_all, occT_all, occD_all, T);
    return id;
}

// pick_first_to for a fill started by carry_ply_start
CCX_HD int carry_ply_to(const JumpFill &f, u32 r1, const TriTables &T)
{
    return select64_step(f.reach, ccx_umulhi(r1, (u32)ccx_popcll(f.reach)), T.sSel);
}

// cells of one diagonal level l = r - c + 6 (human row l + 1)
CCX_HD u64 diag_mask(int l)
{
    const u64 D0 = 0x0040201008040201ULL;            // bits 9r, r = 0..6
    int k = 6 - l;                                   // c = r + k
    if (k >= 0) return (D0 << k) & ((1ULL << (8 * (7 - k))) - 1ULL) & CCX_VALID;
    return (D0 << (8 * (-k))) & CCX_VALID;
}

// GreedyPlayer.decide_move's filtered_best_moves (player.py:99-118) as per-checker destination masks;
// returns the number of candidates.  dist = rows advanced (player.py:103-105); best_moves = max dist;
// last_checker = rearmost start row among them (:113); keep best moves starting on that row (:115).
CCX_HD int greedy_candidates(const Game &g, const u64 (&dest)[6], u64 (&cand)[6])
{
    bool p2 = (g.meta >> 48) & 1;
    int dist[6], start[6];
    int max_dist = -100;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        u32 levels = 0;
#pragma unroll
        for (int l = 0; l < 13; l++) {
            const u64 dm = diag_mask(l);          // constant-folded after unrolling
            levels |= (dest[k] & dm) ? (1u << l) : 0u;
        }
        start[k] = level_of((int)((g.cells_me >> (8 * k)) & 0xFF));
        int best_end = p2 ? (31 - ccx_clz(levels)) : (ccx_ffs(levels) - 1);
        dist[k] = levels ? (p2 ? best_end - start[k] : start[k] - best_end) : -100;
        max_dist = dist[k] > max_dist ? dist[k] : max_dist;
    }
    int s_star = p2 ? 100 : -100;
#pragma unroll
    for (int k = 0; k < 6; k++)
        if (dist[k] == max_dist) s_star = p2 ? (start[k] < s_star ? start[k] : s_star) : (start[k] > s_star ? start[k] : s_star);
    int total = 0;
    if (max_dist == -100) {
#pragma unroll
        for (int k = 0; k < 6; k++) cand[k] = 0;
        return 0;
    }
    u64 end_mask = diag_mask(p2 ? s_star + max_dist : s_star - max_dist);
#pragma unroll
    for (int k = 0; k < 6; k++) {
        cand[k] = (dist[k] == max_dist && start[k] == s_star) ? (dest[k] & end_mask) : 0;
        total += ccx_popcll(cand[k]);
    }
    return total;
}

// uniform pick among the candidates in canonical order (checker id, then ascending cell) — player.py:121
CCX_HD int pick_candidate(const Game &g, const u64 (&cand)[6], int total, u32 r0, int &from, int &to)
{
    int pick = (int)ccx_umulhi(r0, (u32)total);
    int id = 0; u64 m = 0; int base = 0; bool found = false;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        int c = ccx_popcll(cand[k]);
        if (!found && pick < base + c) { id = k; m = cand[k]; pick -= base; found = true; }
        base += c;
    }
    to = select64(m, (u32)pick);
    from = (int)((g.cells_me >> (8 * id)) & 0xFF);
    return id;
}

// game.py:73-82: with 16 stored destinations, the mover's are every second one from the end
CCX_HD bool repetition_stop(u64 lo, u64 hi)
{
    u64 seen = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        seen |= 1ULL << ((lo >> (16 * q)) & 63);
        seen |= 1ULL << ((hi >> (16 * q)) & 63);
    }
    return ccx_popcll(seen) <= 3;                    // config.py:16 UNIQUE_DEST_LIMIT
}

CCX_HD u64 undo_in_cells(u64 cells, int from, int to)
{
#pragma unroll
    for (int k = 0; k < 6; k++)
        if (((cells >> (8 * k)) & 0xFF) == (u64)to) cells = (cells & ~(0xFFULL << (8 * k))) | ((u64)from << (8 * k));
    return cells;
}
