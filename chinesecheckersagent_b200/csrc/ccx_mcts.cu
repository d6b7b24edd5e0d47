// ccx_mcts.cu — batched MCTS (MCTS.py:13-153) as per-tree device node pools, one warp per tree.
//
// Reference semantics kept bit for bit (SURVEY.md §7.4): one simulation at a time per tree, PUCT in
// IEEE float64 evaluated left to right without FMA contraction (MCTS.py:62-63), strict-'>' running
// maximum so the first maximal edge wins (MCTS.py:65-69 with the first-choice tie-break), un-normalised
// priors (MCTS.py:108), terminal leaves never expanded (MCTS.py:81-90), no virtual loss, no tree reuse.  (Opt-in exceptions:
// the leaf-parallel rounds further down select up to L leaves per tree per round under virtual loss; L = 1 is the above.  A reuse
// begin, ccx_mcts_begin_reuse, starts a search from the subtree the previous search grew below the new root.)
// What changes is the machinery: instead of deep-copying a Board into one Node object per legal move
// (MCTS.py:104-107) a tree is a bump-allocated edge pool (SoA: N, W, P, child, move) plus a pool of the
// nodes that were actually visited; a child's 40-byte state is materialised lazily on its first visit.
//
// Edge order = checker id ascending, then destination cell ascending ("canonical", BASELINE.json).
#include "ccx_device.cuh"
#include "ccx_internal.h"
#include "ccx_fpmath.cuh"
#include "ccx_gumbel_table.h"
#include "ccx_sym.cuh"
#include <cfloat>
#include <new>
#include <cmath>
#include <cstdlib>

#define FULL 0xFFFFFFFFu
#define MCTS_WARPS_PER_BLOCK 2
#define NODE_WORDS 6            // 5 state words + info word

// info word of a node: edge_begin (32) | n_edges (8) | spare (16) | winner (4) | expanded (4).  The copy the descent reads lives
// on the parent's edge (eInfo) for every node but the root.
// (Tried and dropped, r01c: keeping N_sum in the spare bits, maintained by the backup, so that sqrt(N_sum) is ready before
// the edge statistics arrive — self-play +0.8 %, stub search -3 %: the extra read-modify-write per level costs what it saves.)
// (Tried and dropped, r01f: an L2 prefetch of the chosen edge's W during the descent, for the backup that reads it — stub search
// 5.49e8 -> 5.35e8 sims/s, self-play ply 18.37 -> 18.60 ms.)
__device__ __forceinline__ u64 make_info(u32 eb, u32 ne, u32 winner, u32 expanded)
{
    return (u64)eb | ((u64)(ne & 0xFF) << 32) | ((u64)(winner & 0xF) << 56) | ((u64)(expanded & 0xF) << 60);
}
__device__ __forceinline__ int info_ne(u64 info) { return (int)((info >> 32) & 0xFF); }
__device__ __forceinline__ int info_eb(u64 info) { return (int)(u32)info; }
__device__ __forceinline__ int info_winner(u64 info) { return (int)((info >> 56) & 0xF); }

struct ccx_trees {
    int64_t cap_trees = 0;
    int32_t nodes_per_tree = 0, edges_per_tree = 0, path_max = 0;
    u64 *node = nullptr;        // [T][NPT][NODE_WORDS]
    u32 *eN = nullptr;          // [T][EPT]
    double *eW = nullptr, *eP = nullptr;
    double *eQ = nullptr;       // W / N as of the last backup (MCTS.py:89,118 store Q the same way): the descent divides once per edge, not twice
    int32_t *eChild = nullptr;  // node index inside the tree or -1
    u64 *eInfo = nullptr;       // [T][EPT] copy of the child node's info word (valid once eChild >= 0): the descent reads it
                                // together with eChild, so a tree level costs two dependent memory round trips, not four
    uint16_t *eMove = nullptr;  // checker id << 8 | destination cell
    int32_t *path = nullptr;    // [T][PATH_MAX] edge indices of the current simulation
    int32_t *tree_meta = nullptr;   // [T][8]: n_nodes, n_edges, overflow, path_len, leaf_node, leaf_kind, selections done, root hash
    size_t bytes = 0;
    // PUCT tie rule (ccx_mcts_set_tiebreak): 0 = first maximal edge, 1 = the reference's epsilon-tie list with a Philox draw
    int32_t tie_mode = 0;       // by value: selects the kernel instantiation (and keys the cached round graph)
    u32 *tie_params = nullptr;  // device u32[4]: Philox key lo/hi, uid0 lo/hi — in memory so that a new seed does not invalidate the graph
    const int64_t *tie_uids = nullptr;   // device, caller-owned (ccx_set_slot_ids): uid of tree i when the batch is compacted, else uid0 + i
};

struct TreeView {
    u64 *node; u32 *eN; double *eW; double *eP; double *eQ; int32_t *eChild; u64 *eInfo; uint16_t *eMove; int32_t *path; int32_t *meta;
    int32_t npt, ept, path_max;
    const u32 *tie; const int64_t *tie_uids; u64 tree_index;
};

__device__ __forceinline__ TreeView tree_view(const ccx_trees &t, int64_t tree)
{
    TreeView v;
    v.node = t.node + tree * t.nodes_per_tree * NODE_WORDS;
    v.eN = t.eN + tree * t.edges_per_tree;
    v.eW = t.eW + tree * t.edges_per_tree;
    v.eP = t.eP + tree * t.edges_per_tree;
    v.eQ = t.eQ + tree * t.edges_per_tree;
    v.eChild = t.eChild + tree * t.edges_per_tree;
    v.eInfo = t.eInfo + tree * t.edges_per_tree;
    v.eMove = t.eMove + tree * t.edges_per_tree;
    v.path = t.path + tree * t.path_max;
    v.meta = t.tree_meta + tree * 8;
    v.npt = t.nodes_per_tree; v.ept = t.edges_per_tree; v.path_max = t.path_max;
    v.tie = t.tie_params; v.tie_uids = t.tie_uids; v.tree_index = (u64)tree;
    return v;
}

enum { META_NNODES = 0, META_NEDGES = 1, META_OVERFLOW = 2, META_PATHLEN = 3, META_LEAF = 4, META_LEAFKIND = 5, META_SELECTS = 6,
       META_SERIAL = 7 };
#define TIE_EPSILON 1e-5        // config.py:36 EPSILON
enum { LEAF_EVAL = 0, LEAF_TERMINAL = 1, LEAF_DEAD = 2 };
enum { EVAL_UNIFORM = 0, EVAL_HASH = 1, EVAL_NET = 2 };

// sqrt of small integers, correctly rounded (filled on the host with IEEE sqrt, which is what the device's sqrt(double) returns
// too): np.sqrt(N_sum) of the descent becomes one broadcast constant load instead of a ~150-cycle dependent sequence per level
#define SQRT_TABLE 1024
__constant__ double c_sqrt[SQRT_TABLE];
__device__ __forceinline__ double sqrt_count(u32 n) { return n < SQRT_TABLE ? c_sqrt[n] : sqrt((double)n); }

__device__ __forceinline__ u64 shfl64(u64 v, int src)
{
    u32 lo = __shfl_sync(FULL, (u32)v, src), hi = __shfl_sync(FULL, (u32)(v >> 32), src);
    return (u64)lo | ((u64)hi << 32);
}

__device__ __forceinline__ Game game_of_words(u64 occ1, u64 occ2, u64 c1, u64 c2, u64 meta)
{
    Game g;
    g.meta = meta;
    bool p2 = (meta >> 48) & 1;
    g.occ_me = p2 ? occ2 : occ1; g.occ_op = p2 ? occ1 : occ2;
    g.cells_me = p2 ? c2 : c1;   g.cells_op = p2 ? c1 : c2;
    return g;
}

__device__ __forceinline__ Game load_node_game(const TreeView &tv, int node)
{
    const u64 *w = tv.node + (int64_t)node * NODE_WORDS;
    return game_of_words(w[0], w[1], w[2], w[3], w[4]);
}

__device__ __forceinline__ void store_node(const TreeView &tv, int node, const Game &g, u64 info)
{
    u64 *w = tv.node + (int64_t)node * NODE_WORDS;
    bool p2 = (g.meta >> 48) & 1;
    w[0] = p2 ? g.occ_op : g.occ_me; w[1] = p2 ? g.occ_me : g.occ_op;
    w[2] = p2 ? g.cells_op : g.cells_me; w[3] = p2 ? g.cells_me : g.cells_op;
    w[4] = g.meta; w[5] = info;
}

// ---- test evaluators (specification shared with the CPU checker; not reference code) ---------------
__host__ __device__ constexpr u64 splitmix64_c(u64 z)
{
    z += 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__host__ __device__ constexpr u64 plane6_sum()
{
    u64 s = 0;
    for (int c = 0; c < 49; c++) s += splitmix64_c((u64)(c * 7 + 6) + 1);
    return s;
}

// hash of utils.to_model_input(state, side to move): sum over non-zero plane entries of
// splitmix64(k+1) * value, k = (r*7+c)*7 + channel.  Warp-cooperative: 36 labelled entries + plane 6.
__device__ __forceinline__ u64 warp_sum_u64(u64 v)
{
#pragma unroll
    for (int off = 16; off; off >>= 1) v += shfl64(v, (threadIdx.x & 31) ^ off);
    return v;
}

__device__ __forceinline__ u64 leaf_hash(const Game &g, int lane)
{
    int plies = (int)((g.meta >> 32) & 0xFFFF);
    u64 cur0 = g.cells_me, opp0 = g.cells_op;
    u64 opp1 = undo_in_cells(opp0, (int)(g.meta & 0xFF), (int)((g.meta >> 8) & 0xFF));
    u64 cur2 = undo_in_cells(cur0, (int)((g.meta >> 16) & 0xFF), (int)((g.meta >> 24) & 0xFF));
    u64 h = 0;
    for (int e = lane; e < 36; e += 32) {
        int hs = e / 12, side = (e / 6) & 1, id = e % 6;
        if (hs > plies) continue;
        u64 cells = side ? (hs >= 1 ? opp1 : opp0) : (hs >= 2 ? cur2 : cur0);
        int cell = (int)((cells >> (8 * id)) & 0xFF);
        int k = ((cell >> 3) * 7 + (cell & 7)) * 7 + 2 * hs + side;
        h += splitmix64_c((u64)k + 1) * (u64)(id + 1);
    }
    h = warp_sum_u64(h);
    if ((g.meta >> 48) & 1) h += plane6_sum();                   // utils.py:157-158
    return h;
}

// ---- select (MCTS.moveToLeaf, MCTS.py:49-76) ---------------------------------------------------------
// Returns the leaf node index (materialising it if this is its first visit) and leaves the path in
// tv.path / path_len.  leaf_kind: LEAF_EVAL (needs evaluation + expansion), LEAF_TERMINAL (winner != 0).
// PREFETCH: fetch the child index and child info word of EVERY edge together with the edge statistics, so that a tree level
// is ONE dependent memory round trip (the chosen edge's pair comes out of a shuffle).  Pays off for the deep, narrow trees a
// real net produces (round-based kernels: -1.9 % per self-play ply); costs bandwidth on the wide, shallow trees of the
// uniform-prior stub (persistent kernel: -19 %), which therefore reads the pair after the arg-max.
// VL (leaf-parallel rounds): the descent sees the virtual losses vl[e] of the round's pending selections — N' = N + V,
// N_sum' = sum N', Q' = (W - V) / (N + V) for V > 0 — while the stored N, W, Q stay the real statistics.
template <bool PREFETCH, bool TIES, bool VL = false>
__device__ __forceinline__ int select_leaf(const TreeView &tv, int lane, double cpuct, int &path_len, int &leaf_kind,
                                           const uint8_t *vl = nullptr)
{
    int node = 0, depth = 0;
    u64 info = tv.node[5];
    // tie rule 1: simulation index and search serial of this tree key the Philox draws (read before lane 0 advances the counter)
    const u32 sim_index = TIES ? (u32)tv.meta[META_SELECTS] : 0u;
    const u32 serial = TIES ? (u32)tv.meta[META_SERIAL] : 0u;
    for (;;) {
        int winner = info_winner(info);
        int ne = info_ne(info);
        if (winner) { leaf_kind = LEAF_TERMINAL; break; }
        if (ne == 0) { leaf_kind = LEAF_EVAL; break; }           // Node.isLeaf()
        int eb = info_eb(info);
        // one pass over the edges: N, W, P of edges lane, lane+32, ... stay in registers (<= 126 legal moves)
        // (tried, r02h: skipping the chunks past the node's last edge with warp-uniform branches — mean branching is 24, one chunk
        // of the four usually suffices — same trees; stub search 1.323 against 1.315 ms, self-play ply 29.6 against 29.0 ms: the
        // predicated-off loads cost less than the branches)
        u32 Nr[4]; double Wr[4], Pr[4]; int Cr[4]; u64 Ir[4]; u32 Vr[4];
        u32 nsum = 0;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            int j = lane + 32 * c;
            bool in = j < ne;
            if (PREFETCH) {
                Cr[c] = in ? tv.eChild[eb + j] : -1;
                Ir[c] = in ? tv.eInfo[eb + j] : 0ULL;
            }
            Nr[c] = in ? tv.eN[eb + j] : 0u;
            Wr[c] = in ? tv.eQ[eb + j] : 0.0;                    // Q = W / N, stored by the backup
            Pr[c] = in ? tv.eP[eb + j] : 0.0;
            if (VL) {
                Vr[c] = in ? (u32)vl[eb + j] : 0u;
                Nr[c] += Vr[c];                                  // N' = N + V
            }
            nsum += Nr[c];
        }
        nsum = __reduce_add_sync(FULL, nsum);                    // N_sum (MCTS.py:58-59)
        double sq = sqrt_count(nsum);                            // np.sqrt(N_sum)
        double best = -INFINITY; int besti = 0x7FFFFFFF;
        double QUr[4];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            int j = lane + 32 * c;
            QUr[c] = -INFINITY;
            if (j < ne) {
                u32 N = Nr[c];
                double Q = Wr[c];                                                               // MCTS.py:89,118
                if (VL && Vr[c]) Q = __ddiv_rn(__dsub_rn(tv.eW[eb + j], (double)Vr[c]), (double)N);   // a loss for the mover
                double U = __ddiv_rn(__dmul_rn(__dmul_rn(cpuct, Pr[c]), sq), __dadd_rn(1.0, (double)N));   // :62
                double QU = __dadd_rn(Q, U);                                                    // :63
                if (TIES) QUr[c] = QU;
                if (QU > best) { best = QU; besti = j; }                                        // :65-67
            }
        }
        // warp arg-max, ties to the smallest edge index (= first maximal edge in list order): order-preserving 64-bit key of
        // the double (no NaNs here; + 0.0 folds a -0.0 into +0.0 so that equal values have equal keys), three warp reductions
        {
            u64 u = (u64)__double_as_longlong(best + 0.0);
            u64 key = (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
            u32 hi = (u32)(key >> 32), lo = (u32)key;
            u32 mhi = __reduce_max_sync(FULL, hi);
            u32 mlo = __reduce_max_sync(FULL, hi == mhi ? lo : 0u);
            besti = (int)__reduce_min_sync(FULL, (hi == mhi && lo == mlo) ? (u32)besti : 0x7FFFFFFFu);
            if (TIES) {
                // MCTS.py:65-72: chosen_edges = [first edge attaining the maximum] + every later edge with fabs(QU - maxQU) < EPSILON
                // (earlier near-ties were dropped by the reset at :66-67); random.choice -> Philox, index = mulhi(x, len)
                const u64 mkey = ((u64)mhi << 32) | mlo;
                const double M = __longlong_as_double((long long)((mkey >> 63) ? (mkey & 0x7FFFFFFFFFFFFFFFULL) : ~mkey));
                u32 cm[4]; int total = 0;
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    int j = lane + 32 * c;
                    bool cand = j < ne && (j == besti || (j > besti && fabs(QUr[c] - M) < TIE_EPSILON));
                    cm[c] = __ballot_sync(FULL, cand);
                    total += __popc(cm[c]);
                }
                if (total > 1) {
                    const u64 uid = tv.tie_uids ? (u64)tv.tie_uids[tv.tree_index] : (((u64)tv.tie[3] << 32) | tv.tie[2]) + tv.tree_index;
                    Philox4 rnd = philox4x32_10(tv.tie[0], tv.tie[1], sim_index, (u32)depth, (u32)uid ^ (serial * 0x9E3779B9u),
                                                (u32)(uid >> 32) ^ 0x7E1Bu);
                    int k = (int)__umulhi(rnd.x, (u32)total);
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        int pc = __popc(cm[c]);
                        if (k >= 0 && k < pc) { besti = 32 * c + (int)__fns(cm[c], 0, k + 1); k = -1; }
                        else if (k >= 0) k -= pc;
                    }
                }
            }
        }
        int e = eb + besti;
        if (lane == 0 && depth < tv.path_max) tv.path[depth] = e;
        depth++;
        int child; u64 cinfo;                                    // cinfo is meaningful iff child >= 0
        if (PREFETCH) {
            const int chunk = besti >> 5, src = besti & 31;
            child = __shfl_sync(FULL, chunk == 0 ? Cr[0] : chunk == 1 ? Cr[1] : chunk == 2 ? Cr[2] : Cr[3], src);
            cinfo = shfl64(chunk == 0 ? Ir[0] : chunk == 1 ? Ir[1] : chunk == 2 ? Ir[2] : Ir[3], src);
        } else {
            child = tv.eChild[e];
            cinfo = tv.eInfo[e];
        }
        if (child < 0) {
            // first visit: materialise the child state = Board.place on a copy (MCTS.py:104-105)
            int nn = tv.meta[META_NNODES];
            if (nn >= tv.npt) { if (lane == 0) tv.meta[META_OVERFLOW] = 1; leaf_kind = LEAF_DEAD; node = 0; break; }
            Game g = load_node_game(tv, node);
            u32 mv = tv.eMove[e];
            int id = (int)(mv >> 8), to = (int)(mv & 0xFF);
            int from = (int)((g.cells_me >> (8 * id)) & 0xFF);
            apply_move(g, id, from, to);
            int w = winner_of(g);
            __syncwarp();
            if (lane == 0) {
                store_node(tv, nn, g, make_info(0, 0, (u32)w, 0));
                tv.eChild[e] = nn;
                tv.eInfo[e] = make_info(0, 0, (u32)w, 0);
                tv.meta[META_NNODES] = nn + 1;
            }
            __syncwarp();
            node = nn;
            leaf_kind = w ? LEAF_TERMINAL : LEAF_EVAL;
            break;
        }
        node = child;
        info = cinfo;
    }
    path_len = depth;
    if (TIES && lane == 0) tv.meta[META_SELECTS] = (int32_t)(sim_index + 1u);
    return node;
}

// ---- backup (MCTS.py:83-90 terminal, 112-118 value) ---------------------------------------------------
__device__ __forceinline__ void backup(const TreeView &tv, int lane, int path_len, double v, bool terminal)
{
    for (int d = lane; d < path_len; d += 32) {
        int e = tv.path[d];
        bool same = ((path_len - d) & 1) == 0;                   // edge.currPlayer == leafNode.currPlayer
        double delta = terminal ? (same ? -1.0 : 1.0)            // REWARD['win'] * direction
                                : __dmul_rn(v, same ? 1.0 : -1.0);
        u32 N = tv.eN[e] + 1;
        double W = __dadd_rn(tv.eW[e], delta);
        tv.eN[e] = N;
        tv.eW[e] = W;
        tv.eQ[e] = __ddiv_rn(W, (double)N);                       // edge.stats['Q'] = W / N
    }
}

// ---- expand (MCTS.py:95-109) ---------------------------------------------------------------------------
// Lanes 0..5 run one checker's flood fill each; the six masks are then broadcast and every lane writes a
// strided share of the edge list.  prior(idx) is supplied by the evaluator functor.
// parent_edge = the edge that leads to `node` (last edge of the path), -1 for the root: its eInfo copy is refreshed.
template <typename PriorFn>
__device__ __forceinline__ bool expand_node(const TreeView &tv, int lane, int node, const Game &g, PriorFn prior, const uint8_t *sT,
                                            int parent_edge)
{
    u64 mine = 0;
    if (lane < 6) {
        u64 occ_all = g.occ_me | g.occ_op;
        u64 o = 1ULL << ((g.cells_me >> (8 * lane)) & 0xFF);
        u64 occ = occ_all & ~o, empty = ~occ & CCX_VALID;
        u64 todo = o, reach = 0;
        while (todo) {                                        // ray expansion of one cell per iteration (ccx_device.cuh)
            int i = 63 - __clzll((long long)todo);         // order-independent closure; top bit = one FLO
            todo ^= 1ULL << i;
            u64 nw = expand_cell(i, occ, sT) & ~(reach | o);
            reach |= nw; todo |= nw;
        }
        mine = (neighbours(o) & empty) | reach;
    }
    u64 dest[6]; int pre[7]; pre[0] = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) { dest[k] = shfl64(mine, k); pre[k + 1] = pre[k] + __popcll(dest[k]); }
    int total = pre[6];
    int eb = tv.meta[META_NEDGES];
    if (eb + total > tv.ept) { if (lane == 0) tv.meta[META_OVERFLOW] = 1; return false; }
    for (int j = lane; j < total; j += 32) {
        int k = 0;
#pragma unroll
        for (int q = 1; q < 6; q++) k += (j >= pre[q]);
        u64 m = 0; int base = 0;
#pragma unroll
        for (int q = 0; q < 6; q++) if (k == q) { m = dest[q]; base = pre[q]; }
        int to = select64(m, (u32)(j - base));
        int idx = k * 49 + (to >> 3) * 7 + (to & 7);             // utils.encode_checker_index
        tv.eN[eb + j] = 0; tv.eW[eb + j] = 0.0; tv.eQ[eb + j] = 0.0; tv.eP[eb + j] = prior(idx);     // MCTS.py:32-37,108
        tv.eChild[eb + j] = -1;
        tv.eMove[eb + j] = (uint16_t)((k << 8) | to);
    }
    __syncwarp();
    if (lane == 0) {
        tv.meta[META_NEDGES] = eb + total;
        u64 *info = tv.node + (int64_t)node * NODE_WORDS + 5;
        *info = make_info((u32)eb, (u32)total, 0, 1);
        if (parent_edge >= 0) tv.eInfo[parent_edge] = make_info((u32)eb, (u32)total, 0, 1);
    }
    __syncwarp();
    return true;
}

struct UniformPrior { __device__ double operator()(int) const { return 1.0 / 294.0; } };
struct HashPrior {
    u32 k0, k1;
    __device__ double operator()(int idx) const { return (double)philox4x32_10(k0, k1, (u32)idx, 7u, 0u, 0u).x / 4294967296.0; }
};
struct TablePrior {      // priors from an evaluator's output row p[294] (float64)
    const double *p;
    __device__ double operator()(int idx) const { return p[idx]; }
};

// evaluate + expand + backup of one leaf with an in-kernel evaluator
template <int EVAL>
__device__ __forceinline__ void eval_expand_backup(const TreeView &tv, int lane, int leaf, int path_len, const uint8_t *sT)
{
    Game g = load_node_game(tv, leaf);
    const int parent_edge = path_len > 0 ? tv.path[path_len - 1] : -1;
    double v = 0.0;
    bool ok;
    if (EVAL == EVAL_HASH) {
        u64 h = leaf_hash(g, lane);
        HashPrior pr = {(u32)h, (u32)(h >> 32)};
        v = (double)philox4x32_10(pr.k0, pr.k1, 294u, 7u, 0u, 0u).x / 2147483648.0 - 1.0;
        ok = expand_node(tv, lane, leaf, g, pr, sT, parent_edge);
    } else {
        ok = expand_node(tv, lane, leaf, g, UniformPrior(), sT, parent_edge);
    }
    if (ok) backup(tv, lane, path_len, v, false);
}

// selfplay.py:121-124 — root priors mixed with caller-supplied Dirichlet noise (one value per root edge)
__device__ __forceinline__ void mix_root_noise(const TreeView &tv, int lane, const double *noise, bool normalize = false)
{
    u64 info = tv.node[5];
    int ne = info_ne(info), eb = info_eb(info);
    double scale = 1.0;
    if (normalize) {                      // raw gamma draws -> Dirichlet sample over the ne root edges
        double sum = 0.0;
        for (int j = lane; j < ne; j += 32) sum += noise[j];
#pragma unroll
        for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
        scale = sum > 0.0 ? 1.0 / sum : 0.0;
    }
    for (int j = lane; j < ne; j += 32) {
        double p = __dmul_rn(tv.eP[eb + j], 1. - 0.25);
        double nz = normalize ? noise[j] * scale : noise[j];
        tv.eP[eb + j] = __dadd_rn(p, __dmul_rn(0.25, nz));
    }
    __syncwarp();
}

// A root whose status is not RUNNING or whose ply count is below min_ply gets an inactive tree
// (META_OVERFLOW = 2): every later phase skips it (self-play: opening random plies, finished games).
__device__ __forceinline__ bool root_inactive(u64 m, int min_ply, int ply_parity)
{
    bool inactive = min_ply >= 0 && ((m >> 56) != 0 || (int)((m >> 32) & 0xFFFF) < min_ply);
    if (ply_parity >= 0 && (int)((m >> 32) & 1) != ply_parity) inactive = true;          // two-net self-play: the other net's plies
    return inactive;
}

// "search serial" of the tie rule: a hash of the root position, so that the draws of a search depend on (seed, tree uid, root)
// only — never on what the handle searched before
__device__ __forceinline__ int32_t root_serial(const u64 *roots, int64_t n, int64_t tree)
{
    u64 z = roots[0 * n + tree] * 0x9E3779B97F4A7C15ULL + roots[1 * n + tree] * 0xC2B2AE3D27D4EB4FULL +
            (roots[4 * n + tree] & 0x0000FFFFFFFFFFFFULL);
    return (int32_t)((u32)(z >> 32) ^ (u32)z);
}

__device__ __forceinline__ void init_tree(const TreeView &tv, int lane, const u64 *roots, int64_t n, int64_t tree, int min_ply = 0,
                                          int ply_parity = -1)
{
    if (lane == 0) {
        const bool inactive = root_inactive(roots[4 * n + tree], min_ply, ply_parity);
        tv.meta[META_SELECTS] = 0;
        tv.meta[META_SERIAL] = root_serial(roots, n, tree);
        Game g = game_of_words(roots[0 * n + tree], roots[1 * n + tree], roots[2 * n + tree], roots[3 * n + tree],
                               roots[4 * n + tree] & 0x00FFFFFFFFFFFFFFULL);
        store_node(tv, 0, g, make_info(0, 0, (u32)winner_of(g), 0));
        tv.meta[META_NNODES] = 1; tv.meta[META_NEDGES] = 0; tv.meta[META_OVERFLOW] = inactive ? 2 : 0; tv.meta[META_PATHLEN] = 0;
    }
    __syncwarp();
}

// Persistent search with an in-kernel evaluator: every warp runs all simulations of its tree.
// select_leaf<PREFETCH> in the persistent kernel: measured again in r02 under the 72-register cap (one resident wave): 1.321 ms
// per 4,096-tree search with the prefetch against 1.310 ms without (round 1 saw -19 % because 84 registers split the launch
// into 1.15 waves).  No gain either way: at 1,100 warp instructions per simulation and 59 % issue utilisation the kernel is as
// much instruction- as latency-bound.
#ifndef CCX_SEARCH_PREFETCH
#define CCX_SEARCH_PREFETCH false
#endif
template <int EVAL, bool TIES>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_search(ccx_trees trees, const u64 *__restrict__ roots, int64_t n, int num_itr, double cpuct, int pre_expand,
              const double *__restrict__ noise, int noise_stride, const uint8_t *__restrict__ jt)
{
    __shared__ __align__(16) uint8_t sT[CCX_JT_BYTES];
    for (int q = threadIdx.x; q < CCX_JT_BYTES / 16; q += blockDim.x) reinterpret_cast<uint4 *>(sT)[q] = reinterpret_cast<const uint4 *>(jt)[q];
    __syncthreads();
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    init_tree(tv, lane, roots, n, tree, -1);
    if (pre_expand && info_winner(tv.node[5]) == 0) {                    // selfplay.py:117
        eval_expand_backup<EVAL>(tv, lane, 0, 0, sT);
        if (noise) mix_root_noise(tv, lane, noise + tree * noise_stride);
    }
    if (pre_expand && TIES && lane == 0) tv.meta[META_SELECTS] = 1;      // the round-based drivers spend selection 0 on the root expansion
    __syncwarp();
    for (int it = 0; it < num_itr; it++) {                                   // MCTS.py:123-125
        int path_len, kind;
        int leaf = select_leaf<CCX_SEARCH_PREFETCH, TIES>(tv, lane, cpuct, path_len, kind);
        __syncwarp();
        if (kind == LEAF_TERMINAL) backup(tv, lane, path_len, 0.0, true);
        else if (kind == LEAF_EVAL) eval_expand_backup<EVAL>(tv, lane, leaf, path_len, sT);
        __syncwarp();
        if (tv.meta[META_OVERFLOW]) break;
    }
}

// ---- round-based pieces for an external evaluator (the policy/value net) ----------------------------
// phase A: select one leaf per tree; terminal leaves are backed up at once; for the others the leaf's
// state words are written to leaf_state[5][n] (input of ccx_encode / the net)
template <bool TIES>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_select(ccx_trees trees, int64_t n, double cpuct, u64 *__restrict__ leaf_state)
{
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    if (tv.meta[META_OVERFLOW]) {
        // inactive / overflowed tree: hand the evaluator a well-formed dummy position (its output is ignored)
        if (lane == 0) {
            tv.meta[META_LEAFKIND] = LEAF_DEAD;
            leaf_state[0 * n + tree] = CCX_START_OCC1; leaf_state[1 * n + tree] = CCX_START_OCC2;
            leaf_state[2 * n + tree] = CCX_START_CELLS1; leaf_state[3 * n + tree] = CCX_START_CELLS2;
            leaf_state[4 * n + tree] = CCX_START_META;
        }
        return;
    }
    int path_len, kind;
    int leaf = select_leaf<true, TIES>(tv, lane, cpuct, path_len, kind);
    __syncwarp();
    if (kind == LEAF_TERMINAL) backup(tv, lane, path_len, 0.0, true);
    if (lane < 5) leaf_state[lane * n + tree] = tv.node[(int64_t)leaf * NODE_WORDS + lane];
    if (lane == 0) { tv.meta[META_PATHLEN] = path_len; tv.meta[META_LEAF] = leaf; tv.meta[META_LEAFKIND] = kind; }
}

// phase B: expand the selected leaf with priors p[n][294] (float64, already soft-maxed: model.py:21-24)
// and back up v[n]; root_only_noise != NULL mixes Dirichlet noise into the root priors (first call).
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_expand_backup(ccx_trees trees, int64_t n, const double *__restrict__ p, const double *__restrict__ v,
                     const double *__restrict__ noise, int noise_stride, int noise_normalize, const uint8_t *__restrict__ jt)
{
    __shared__ __align__(16) uint8_t sT[CCX_JT_BYTES];
    for (int q = threadIdx.x; q < CCX_JT_BYTES / 16; q += blockDim.x) reinterpret_cast<uint4 *>(sT)[q] = reinterpret_cast<const uint4 *>(jt)[q];
    __syncthreads();
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    if (tv.meta[META_LEAFKIND] != LEAF_EVAL) return;
    int leaf = tv.meta[META_LEAF], path_len = tv.meta[META_PATHLEN];
    Game g = load_node_game(tv, leaf);
    TablePrior pr = {p + tree * CCX_NUM_ACTIONS};
    if (expand_node(tv, lane, leaf, g, pr, sT, path_len > 0 ? tv.path[path_len - 1] : -1)) backup(tv, lane, path_len, v[tree], false);
    if (noise && leaf == 0) mix_root_noise(tv, lane, noise + tree * noise_stride, noise_normalize != 0);
}

// ---- fused round pieces for the built-in net evaluator (ccx_mcts_run_net) -------------------------------
// phase A': select + utils.to_model_input of the leaf (utils.py:101-160) written straight into the net's uint8
// input batch, one warp per tree (the leaf's 343 bytes are staged in shared memory: zero, scatter the 36
// labels, copy out).  SYM != SYM_OFF (ccx_net_set_symmetry): the leaf's rows in that mode's layout, dst = row tree * SymRows,
// orientation key (k0, k1).
template <bool TIES, int SYM = SYM_OFF>
__device__ __forceinline__ void do_select_encode(const TreeView &tv, int lane, double cpuct, uint8_t *__restrict__ sp,
                                                 uint8_t *__restrict__ dst, u32 k0 = 0, u32 k1 = 0)
{
    Game g;
    if (tv.meta[META_OVERFLOW]) {
        // inactive / overflowed tree: hand the evaluator a well-formed dummy position (its output is ignored)
        if (lane == 0) tv.meta[META_LEAFKIND] = LEAF_DEAD;
        reset_start(g);
    } else {
        int path_len, kind;
        int leaf = select_leaf<true, TIES>(tv, lane, cpuct, path_len, kind);
        __syncwarp();
        if (kind == LEAF_TERMINAL) backup(tv, lane, path_len, 0.0, true);
        if (lane == 0) { tv.meta[META_PATHLEN] = path_len; tv.meta[META_LEAF] = leaf; tv.meta[META_LEAFKIND] = kind; }
        g = load_node_game(tv, leaf);
    }
    if constexpr (SYM != SYM_OFF) {
        sym_encode<SYM>(g, lane, k0, k1, sp, dst);
    } else {
        for (int i = lane; i < 88; i += 32) reinterpret_cast<uint32_t *>(sp)[i] = 0u;
        __syncwarp();
        {
            const int plies = (int)((g.meta >> 32) & 0xFFFF);
            const u64 cur0 = g.cells_me, opp0 = g.cells_op;
            const u64 opp1 = undo_in_cells(opp0, (int)(g.meta & 0xFF), (int)((g.meta >> 8) & 0xFF));
            const u64 cur2 = undo_in_cells(cur0, (int)((g.meta >> 16) & 0xFF), (int)((g.meta >> 24) & 0xFF));
            for (int e = lane; e < 36; e += 32) {
                int hs = e / 12, side = (e / 6) & 1, id = e % 6;
                if (hs > plies) continue;
                u64 cells = side ? (hs >= 1 ? opp1 : opp0) : (hs >= 2 ? cur2 : cur0);
                int c = (int)((cells >> (8 * id)) & 0xFF);
                if (c < 55 && (c & 7) < 7) sp[((c >> 3) * 7 + (c & 7)) * 7 + 2 * hs + side] = (uint8_t)(id + 1);
            }
            if ((g.meta >> 48) & 1)
                for (int c = lane; c < 49; c += 32) sp[c * 7 + 6] = 1;                // utils.py:157-158
        }
        __syncwarp();
        for (int i = lane; i < 343; i += 32) dst[i] = sp[i];
    }
}

template <bool TIES>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_select_encode(ccx_trees trees, int64_t tree0, int64_t n, double cpuct, uint8_t *__restrict__ planes)
{
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);      // trees [tree0, tree0 + n)
    int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    do_select_encode<TIES>(tv, lane, cpuct, sP[threadIdx.x >> 5], planes + tree * 343);
}

// phase B': float64 softmax over all 294 logits (model.py:21-24, utils.py:187-192; same arithmetic as
// k_softmax_f64) + expand + backup, one warp per tree; the priors never touch global memory.  SYM != SYM_OFF: lg = the leaf's
// SymRows rows, priors as ccx_net_eval takes them in that mode (sym_priors), v = its value (sym_value).
template <int SYM = SYM_OFF>
__device__ __forceinline__ void do_softmax_expand_backup(const TreeView &tv, int lane, const float *__restrict__ lg, double v,
                                                         const double *__restrict__ noise, int noise_normalize, double *__restrict__ pr,
                                                         const uint8_t *__restrict__ sT, u32 k0 = 0, u32 k1 = 0)
{
    if (tv.meta[META_LEAFKIND] != LEAF_EVAL) return;
    if (SYM != SYM_OFF) {
        const u64 *w = tv.node + (int64_t)tv.meta[META_LEAF] * NODE_WORDS;
        sym_priors<SYM>(lane, lg, SYM == SYM_RANDOM && sym_mirrored(k0, k1, w[0], w[1], w[4]), pr);
    } else {
        double x[10], mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < 10; j++) {
            int i = lane + 32 * j;
            x[j] = i < 294 ? (double)lg[i] : -INFINITY;
            mx = fmax(mx, x[j]);
        }
#pragma unroll
        for (int off = 16; off; off >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, off));
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < 10; j++) { x[j] = (lane + 32 * j) < 294 ? exp(x[j] - mx) : 0.0; sum += x[j]; }
#pragma unroll
        for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
#pragma unroll
        for (int j = 0; j < 10; j++) if (lane + 32 * j < 294) pr[lane + 32 * j] = x[j] / sum;
    }
    __syncwarp();
    int leaf = tv.meta[META_LEAF], path_len = tv.meta[META_PATHLEN];
    Game g = load_node_game(tv, leaf);
    TablePrior tp = {pr};
    if (expand_node(tv, lane, leaf, g, tp, sT, path_len > 0 ? tv.path[path_len - 1] : -1)) backup(tv, lane, path_len, v, false);
    if (noise && leaf == 0) mix_root_noise(tv, lane, noise, noise_normalize != 0);
}

__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_softmax_expand_backup(ccx_trees trees, int64_t tree0, int64_t n, const float *__restrict__ logits, const float *__restrict__ value,
                             const double *__restrict__ noise, int noise_stride, int noise_normalize, const uint8_t *__restrict__ jt)
{
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    const uint8_t *sT = jt;          // one expansion per launch: the 6 KB jump table is read through L1 instead of staged per block
    int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    do_softmax_expand_backup(tv, lane, logits + tree * 294, (double)value[tree], noise ? noise + tree * noise_stride : nullptr,
                             noise_normalize, sPr[threadIdx.x >> 5], sT);
}

// one launch per round in steady state: finish the previous round's leaf (softmax + expand + backup), then select and encode
// the next one — the same warp owns the tree in both halves, so the halves need no grid-wide ordering between them
// launch bound: 14 blocks per SM (<= 72 registers) keeps all 2,048 blocks of a 4,096-tree round resident in ONE wave (148 x 14 =
// 2,072); at 80 registers (12 blocks per SM) the last 272 blocks start only when others finish: 1.15 waves, slowest SM 88.6 K cycles
// against 59.7 K on average (profiles/r02b_kernels_ncu.md)
template <bool TIES>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_round(ccx_trees trees, int64_t tree0, int64_t n, double cpuct, const float *__restrict__ logits, const float *__restrict__ value,
             const double *__restrict__ noise, int noise_stride, int noise_normalize, uint8_t *__restrict__ planes,
             const uint8_t *__restrict__ jt)
{
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    const uint8_t *sT = jt;          // one expansion per launch: the 6 KB jump table is read through L1 instead of staged per block
    int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    do_softmax_expand_backup(tv, lane, logits + tree * 294, (double)value[tree], noise ? noise + tree * noise_stride : nullptr,
                             noise_normalize, sPr[threadIdx.x >> 5], sT);
    __syncwarp();
    __threadfence_block();
    do_select_encode<TIES>(tv, lane, cpuct, sP[threadIdx.x >> 5], planes + tree * 343);
}

// the three launches above with a mirror-symmetric net evaluation (ccx_net_set_symmetry): tree i owns net rows
// [i * SymRows, (i + 1) * SymRows); (k0, k1) = the random orientation's key
template <bool TIES, int SYM>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_select_encode_sym(ccx_trees trees, int64_t tree0, int64_t n, double cpuct, uint8_t *__restrict__ planes, u32 k0, u32 k1)
{
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    do_select_encode<TIES, SYM>(tv, lane, cpuct, sP[threadIdx.x >> 5], planes + tree * SymRows<SYM>::value * 343, k0, k1);
}

template <bool TIES, int SYM>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_round_sym(ccx_trees trees, int64_t tree0, int64_t n, double cpuct, const float *__restrict__ logits, const float *__restrict__ value,
                 const double *__restrict__ noise, int noise_stride, int noise_normalize, uint8_t *__restrict__ planes,
                 const uint8_t *__restrict__ jt, u32 k0, u32 k1)
{
    constexpr int R = SymRows<SYM>::value;
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    do_softmax_expand_backup<SYM>(tv, lane, logits + tree * R * 294, sym_value<SYM>(value + tree * R),
                                  noise ? noise + tree * noise_stride : nullptr, noise_normalize, sPr[threadIdx.x >> 5], jt, k0, k1);
    __syncwarp();
    __threadfence_block();
    do_select_encode<TIES, SYM>(tv, lane, cpuct, sP[threadIdx.x >> 5], planes + tree * R * 343, k0, k1);
}

template <int SYM>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_softmax_expand_backup_sym(ccx_trees trees, int64_t tree0, int64_t n, const float *__restrict__ logits,
                                 const float *__restrict__ value, const double *__restrict__ noise, int noise_stride, int noise_normalize,
                                 const uint8_t *__restrict__ jt, u32 k0, u32 k1)
{
    constexpr int R = SymRows<SYM>::value;
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    do_softmax_expand_backup<SYM>(tv, lane, logits + tree * R * 294, sym_value<SYM>(value + tree * R),
                                  noise ? noise + tree * noise_stride : nullptr, noise_normalize, sPr[threadIdx.x >> 5], jt, k0, k1);
}

__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_init(ccx_trees trees, const u64 *__restrict__ roots, int64_t n, int min_ply, int ply_parity)
{
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    init_tree(tv, threadIdx.x & 31, roots, n, tree, min_ply, ply_parity);
}

// ---- tree reuse (ccx_mcts_begin_reuse): the subtree of the node that matches the new root becomes the new tree ------------
// Three launches: match (find the node in the source tree), gather (copy its subtree out of place into a
// scratch pool, BFS order, edge ranges / eChild / eInfo remapped, root noise mixed), commit (scratch -> the tree's own slot,
// or a fresh tree).  Out of place, so that any source map (several trees reading one source, a tree reading a slot that is
// rewritten in the same call) is safe.  Per tree rec[4]: source tree, matched node (after the gather: node count), kind
// (1 / 2 = depth of the match, 0 = fresh, -2 = inactive), edge count.
#define STATE_MASK4 0x00FFFFFFFFFFFFFFULL       // META without its status byte (init_tree stores the root so)

// the materialised child of `info`'s node whose state words are w[0..4], or -1
__device__ __forceinline__ int find_child(const TreeView &tv, int lane, u64 info, const u64 *w)
{
    const int ne = info_ne(info), eb = info_eb(info);
    for (int base = 0; base < ne; base += 32) {
        const int j = base + lane;
        const int c = j < ne ? tv.eChild[eb + j] : -1;
        bool hit = false;
        if (c >= 0) {
            const u64 *s = tv.node + (int64_t)c * NODE_WORDS;
            hit = s[0] == w[0] && s[1] == w[1] && s[2] == w[2] && s[3] == w[3] && (s[4] & STATE_MASK4) == w[4];
        }
        const u32 b = __ballot_sync(FULL, hit);
        if (b) return __shfl_sync(FULL, c, __ffs(b) - 1);
    }
    return -1;
}

__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_reuse_match(ccx_trees trees, const u64 *__restrict__ roots, int64_t n, int64_t n_prev, const int64_t *__restrict__ prev,
                   int min_ply, int ply_parity, int64_t lim_visits, int32_t *__restrict__ rec)
{
    const int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= n) return;
    int64_t src = prev ? prev[tree] : tree;
    int node = -1, kind = root_inactive(roots[4 * n + tree], min_ply, ply_parity) ? -2 : 0;
    if (kind == 0 && src >= 0 && src < n_prev) {
        const TreeView sv = tree_view(trees, src);
        if (sv.meta[META_OVERFLOW] == 0) {
            u64 w[5];
#pragma unroll
            for (int k = 0; k < 5; k++) w[k] = roots[k * n + tree];
            w[4] &= STATE_MASK4;
            // every move adds one ply, so the ply counters say at which depth a match can lie
            const int depth = (int)((w[4] >> 32) & 0xFFFF) - (int)((sv.node[4] >> 32) & 0xFFFF);
            const u64 rinfo = sv.node[5];
            if (depth == 1) node = find_child(sv, lane, rinfo, w);
            else if (depth == 2) {
                const int ne = info_ne(rinfo), eb = info_eb(rinfo);
                for (int j = 0; j < ne && node < 0; j++) {
                    const int c = sv.eChild[eb + j];
                    if (c >= 0) node = find_child(sv, lane, sv.eInfo[eb + j], w);
                }
            }
            if (node >= 0) {
                const u64 info = sv.node[(int64_t)node * NODE_WORDS + 5];
                const int ne = info_ne(info), eb = info_eb(info);
                u32 nsum = 0;
                for (int j = lane; j < ne; j += 32) nsum += sv.eN[eb + j];
                nsum = __reduce_add_sync(FULL, nsum);
                if (ne == 0 || (int64_t)nsum > lim_visits) node = -1;          // unexpanded, or more visits than the carry allows
                else kind = depth;
            }
        }
    }
    if (lane == 0) {
        int32_t *r = rec + 4 * tree;
        r[0] = (int32_t)src; r[1] = node; r[2] = kind; r[3] = 0;
    }
}

__device__ __forceinline__ u64 info_rebase(u64 info, int eb) { return (info & 0xFFFFFFFF00000000ULL) | (u32)eb; }

// BFS copy of the matched subtree: the destination node array is the queue (qsrc[q] = source index of destination node q);
// a node's edges are allocated when it is enqueued, so its parent's eInfo copy gets the final edge range at once.  A subtree of
// more than lim_nodes nodes or lim_edges edges falls back to a fresh tree.
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_reuse_gather(ccx_trees trees, ccx_trees scratch, int32_t *__restrict__ qsrc, int64_t n, int32_t *__restrict__ rec, int lim_nodes,
                    int lim_edges, const double *__restrict__ noise, int noise_stride, int noise_normalize)
{
    const int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= n) return;
    int32_t *r = rec + 4 * tree;
    if (r[2] <= 0) return;
    const TreeView sv = tree_view(trees, r[0]), dv = tree_view(scratch, tree);
    int32_t *qs = qsrc + tree * scratch.nodes_per_tree;
    const int m = r[1];
    const u64 rinfo = sv.node[(int64_t)m * NODE_WORDS + 5];
    int qtail = 1, etail = info_ne(rinfo);
    bool ok = qtail <= lim_nodes && etail <= lim_edges;
    if (ok) {
        if (lane < 5) dv.node[lane] = sv.node[(int64_t)m * NODE_WORDS + lane];
        if (lane == 5) dv.node[5] = info_rebase(rinfo, 0);
        if (lane == 0) qs[0] = m;
    }
    __syncwarp();
    for (int q = 0; ok && q < qtail; q++) {
        const int s = qs[q];
        const u64 sinfo = sv.node[(int64_t)s * NODE_WORDS + 5];
        const int ne = info_ne(sinfo), seb = info_eb(sinfo), deb = info_eb(dv.node[(int64_t)q * NODE_WORDS + 5]);
        for (int base = 0; base < ne; base += 32) {
            const int j = base + lane;
            const bool in = j < ne;
            const int c = in ? sv.eChild[seb + j] : -1;
            const bool mat = c >= 0;
            const u64 ci = mat ? sv.eInfo[seb + j] : 0ULL;
            const u32 bal = __ballot_sync(FULL, mat);
            const int rank = __popc(bal & ((1u << lane) - 1u)), nmat = __popc(bal);
            const int cne = mat ? info_ne(ci) : 0;
            int inc = cne;                                                       // inclusive scan of the children's edge counts
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int t = __shfl_up_sync(FULL, inc, off);
                if (lane >= off) inc += t;
            }
            const int esum = __shfl_sync(FULL, inc, 31);
            if (qtail + nmat > lim_nodes || etail + esum > lim_edges) { ok = false; break; }
            if (in) {
                const int k = deb + j, e = seb + j;
                dv.eN[k] = sv.eN[e]; dv.eW[k] = sv.eW[e]; dv.eP[k] = sv.eP[e]; dv.eQ[k] = sv.eQ[e]; dv.eMove[k] = sv.eMove[e];
                const int nc = mat ? qtail + rank : -1;
                const u64 ni = mat ? info_rebase(ci, etail + inc - cne) : 0ULL;
                dv.eChild[k] = nc;
                dv.eInfo[k] = ni;
                if (mat) {
                    const u64 *sw = sv.node + (int64_t)c * NODE_WORDS;
                    u64 *dw = dv.node + (int64_t)nc * NODE_WORDS;
                    dw[0] = sw[0]; dw[1] = sw[1]; dw[2] = sw[2]; dw[3] = sw[3]; dw[4] = sw[4]; dw[5] = ni;
                    qs[nc] = c;
                }
            }
            qtail += nmat; etail += esum;
            __syncwarp();
        }
    }
    if (!ok) { if (lane == 0) r[2] = 0; return; }
    if (lane == 0) { r[1] = qtail; r[3] = etail; }
    __syncwarp();
    if (noise) mix_root_noise(dv, lane, noise + tree * noise_stride, noise_normalize != 0);     // as the round loop's root expansion
}

// scratch -> tree slot for a carried tree (fresh per-search bookkeeping), init_tree for every other; one CTA of
// REUSE_COMMIT_THREADS per tree, a pure copy (measured with one warp per tree: 1.43 ms per 4,096-tree ply)
#define REUSE_COMMIT_THREADS 256
__global__ void __launch_bounds__(REUSE_COMMIT_THREADS)
k_mcts_reuse_commit(ccx_trees trees, ccx_trees scratch, const u64 *__restrict__ roots, int64_t n, const int32_t *__restrict__ rec,
                    int min_ply, int ply_parity, int32_t *__restrict__ reused)
{
    const int64_t tree = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const int32_t *r = rec + 4 * tree;
    const int kind = r[2];
    const TreeView tv = tree_view(trees, tree);
    if (kind <= 0) { if (threadIdx.x < 32) init_tree(tv, lane, roots, n, tree, min_ply, ply_parity); }
    else {
        const TreeView dv = tree_view(scratch, tree);
        const int nn = r[1], ne = r[3];
        for (int i = threadIdx.x; i < nn * NODE_WORDS; i += REUSE_COMMIT_THREADS) tv.node[i] = dv.node[i];
        for (int k = threadIdx.x; k < ne; k += REUSE_COMMIT_THREADS) {
            tv.eN[k] = dv.eN[k]; tv.eW[k] = dv.eW[k]; tv.eP[k] = dv.eP[k]; tv.eQ[k] = dv.eQ[k];
            tv.eChild[k] = dv.eChild[k]; tv.eInfo[k] = dv.eInfo[k]; tv.eMove[k] = dv.eMove[k];
        }
        if (threadIdx.x == 0) {
            tv.meta[META_SELECTS] = 0; tv.meta[META_SERIAL] = root_serial(roots, n, tree);
            tv.meta[META_NNODES] = nn; tv.meta[META_NEDGES] = ne; tv.meta[META_OVERFLOW] = 0; tv.meta[META_PATHLEN] = 0;
        }
    }
    if (reused && threadIdx.x == 0) reused[tree] = kind;
}

// ---- leaf-parallel rounds (ccx_mcts_*_leaves): up to L selections per tree per round under virtual loss -------------
// One CTA of L warps per tree.  Select: warp 0 makes the round's m descents one after another (m = 1 while the root is
// unexpanded, else min(L, selections left in this call)); a pending selection (a non-terminal leaf) adds one virtual loss
// to every edge of its path, which the next descents see; a terminal leaf is backed up at once; a leaf node already chosen
// by a pending selection of this round is a duplicate and is not evaluated.  Then warp k writes evaluator slot k (the
// leaf, or the start position when slot k has nothing to evaluate).  Backup: warp k expands its first-occurrence leaf,
// edge ranges handed out in slot order; then warp 0 walks the pending paths in slot order, removing one virtual loss per
// edge and applying the usual backup (a duplicate with its first occurrence's value).  The virtual losses are zero again
// after every backup phase, overflowed trees included, so no state carries over into the next round or search.
struct ccx_leaf_pool {
    int32_t cap_leaves = 0, path_max = 0;
    int32_t *path = nullptr;    // [T][L][path_max] paths of the round's selections
    int32_t *rec = nullptr;     // [T][L][4] per selection: leaf node, path length, kind (LK_*), first occurrence of a duplicate
    int32_t *meta = nullptr;    // [T][2]: selections made in the current round, selections left in this call
    uint8_t *vl = nullptr;      // [T][EPT] virtual losses of the pending selections through each edge (<= 16)
    size_t bytes = 0;           // (sized for the current trees: a reallocation of the trees frees the pool)
};
enum { LK_NONE = 0, LK_TERMINAL = 1, LK_FIRST = 2, LK_DUP = 3 };

struct LeafView { int32_t *path; int32_t *rec; int32_t *meta; uint8_t *vl; int path_max; };

__device__ __forceinline__ LeafView leaf_view(const ccx_trees &t, const ccx_leaf_pool &lp, int64_t tree)
{
    LeafView v;
    v.path = lp.path + tree * lp.cap_leaves * lp.path_max;
    v.rec = lp.rec + tree * lp.cap_leaves * 4;
    v.meta = lp.meta + tree * 2;
    v.vl = lp.vl + tree * t.edges_per_tree;
    v.path_max = lp.path_max;
    return v;
}

// utils.to_model_input of g into dst[343] (staged in sp[352]: zero, scatter the 36 labels, copy out) — as do_select_encode
__device__ __forceinline__ void encode_planes(const Game &g, int lane, uint8_t *__restrict__ sp, uint8_t *__restrict__ dst)
{
    for (int i = lane; i < 88; i += 32) reinterpret_cast<uint32_t *>(sp)[i] = 0u;
    __syncwarp();
    const int plies = (int)((g.meta >> 32) & 0xFFFF);
    const u64 cur0 = g.cells_me, opp0 = g.cells_op;
    const u64 opp1 = undo_in_cells(opp0, (int)(g.meta & 0xFF), (int)((g.meta >> 8) & 0xFF));
    const u64 cur2 = undo_in_cells(cur0, (int)((g.meta >> 16) & 0xFF), (int)((g.meta >> 24) & 0xFF));
    for (int e = lane; e < 36; e += 32) {
        int hs = e / 12, side = (e / 6) & 1, id = e % 6;
        if (hs > plies) continue;
        u64 cells = side ? (hs >= 1 ? opp1 : opp0) : (hs >= 2 ? cur2 : cur0);
        int c = (int)((cells >> (8 * id)) & 0xFF);
        if (c < 55 && (c & 7) < 7) sp[((c >> 3) * 7 + (c & 7)) * 7 + 2 * hs + side] = (uint8_t)(id + 1);
    }
    if ((g.meta >> 48) & 1)
        for (int c = lane; c < 49; c += 32) sp[c * 7 + 6] = 1;                    // utils.py:157-158
    __syncwarp();
    for (int i = lane; i < 343; i += 32) dst[i] = sp[i];
}

// select phase; budget >= 0 starts a call with that many selections.  ENCODE: slot k -> planes[slot][343] (SYM != SYM_OFF:
// rows [slot * SymRows, (slot + 1) * SymRows) in that mode's layout), else the leaf's state words -> leaf_state[5][n_slots]
template <bool TIES, bool ENCODE, int SYM = SYM_OFF>
__device__ __forceinline__ void leaves_select(const TreeView &tv, const LeafView &lv, int64_t tree, int L, double cpuct, int budget,
                                              uint8_t *__restrict__ planes, u64 *__restrict__ leaf_state, int64_t n_slots,
                                              uint8_t *__restrict__ sp, u32 k0 = 0, u32 k1 = 0)
{
    __shared__ int s_leaf[CCX_MAX_LEAVES], s_kind[CCX_MAX_LEAVES];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (w == 0) {
        int left = budget >= 0 ? budget : lv.meta[1];
        int m = tv.meta[META_OVERFLOW] ? 0 : info_ne(tv.node[5]) == 0 ? 1 : L;     // one selection while the root is unexpanded
        if (m > left) m = left;
        int made = 0;
        for (int k = 0; k < m; k++) {
            TreeView tk = tv;
            tk.path = lv.path + k * lv.path_max;
            int path_len, kind;
            int leaf = select_leaf<true, TIES, true>(tk, lane, cpuct, path_len, kind, lv.vl);
            __syncwarp();
            if (kind == LEAF_DEAD) break;                        // node pool full: the tree is flagged, later phases skip it
            made++;
            int lk = LK_TERMINAL, dup = -1;
            if (kind == LEAF_TERMINAL) backup(tk, lane, path_len, 0.0, true);
            else {
                for (int j = 0; j < k && dup < 0; j++) if (s_kind[j] == LK_FIRST && s_leaf[j] == leaf) dup = j;
                lk = dup < 0 ? LK_FIRST : LK_DUP;
                for (int d = lane; d < path_len; d += 32) lv.vl[tk.path[d]] += 1;       // virtual loss on the pending path
            }
            if (lane == 0) {
                s_leaf[k] = leaf; s_kind[k] = lk;
                int32_t *r = lv.rec + 4 * k;
                r[0] = leaf; r[1] = path_len; r[2] = lk; r[3] = dup;
            }
            __syncwarp();
        }
        for (int k = made + lane; k < L; k += 32) s_kind[k] = LK_NONE;
        if (lane == 0) { lv.meta[0] = made; lv.meta[1] = left - made; }
    }
    __syncthreads();
    if (w < L) {
        const int64_t slot = tree * L + w;
        const bool real = s_kind[w] == LK_FIRST;
        if (ENCODE) {
            Game g;
            if (real) g = load_node_game(tv, s_leaf[w]);
            else reset_start(g);
            if (SYM != SYM_OFF) sym_encode<SYM>(g, lane, k0, k1, sp, planes + slot * SymRows<SYM>::value * 343);
            else encode_planes(g, lane, sp, planes + slot * 343);
        } else if (lane < 5) {
            const u64 dummy = lane == 0 ? CCX_START_OCC1 : lane == 1 ? CCX_START_OCC2 : lane == 2 ? CCX_START_CELLS1
                            : lane == 3 ? CCX_START_CELLS2 : CCX_START_META;
            leaf_state[lane * n_slots + slot] = real ? tv.node[(int64_t)s_leaf[w] * NODE_WORDS + lane] : dummy;
        }
    }
}

// backup phase.  NET: priors = float64 softmax of the float logits (as do_softmax_expand_backup), value float (SYM != SYM_OFF:
// SymRows rows per slot, sym_priors / sym_value); else priors p[slot][294] and v[slot] in float64
template <bool NET, int SYM = SYM_OFF>
__device__ __forceinline__ void leaves_backup(const TreeView &tv, const LeafView &lv, int64_t tree, int L, const void *pv,
                                              const void *vv, const double *__restrict__ noise, int noise_normalize,
                                              double *__restrict__ sPr, const uint8_t *__restrict__ sT, u32 k0 = 0, u32 k1 = 0)
{
    __shared__ int s_cnt[CCX_MAX_LEAVES], s_off[CCX_MAX_LEAVES], s_ov;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m = lv.meta[0];
    const int ov0 = tv.meta[META_OVERFLOW];
    const int64_t slot = tree * L + w;
    int leaf = 0, plen = 0, kind = LK_NONE;
    if (w < m) { leaf = lv.rec[4 * w]; plen = lv.rec[4 * w + 1]; kind = lv.rec[4 * w + 2]; }
    const bool mine = !ov0 && kind == LK_FIRST;
    // (1) priors and legal moves of this warp's leaf
    u64 dest[6]; int pre[7]; pre[0] = 0;
    Game g;
    if (mine) {
        if (NET && SYM != SYM_OFF) {
            const u64 *lw = tv.node + (int64_t)leaf * NODE_WORDS;
            sym_priors<SYM>(lane, (const float *)pv + slot * SymRows<SYM>::value * CCX_NUM_ACTIONS,
                            SYM == SYM_RANDOM && sym_mirrored(k0, k1, lw[0], lw[1], lw[4]), sPr);
        } else if (NET) {
            const float *lg = (const float *)pv + slot * CCX_NUM_ACTIONS;
            double x[10], mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < 10; j++) {
                int i = lane + 32 * j;
                x[j] = i < 294 ? (double)lg[i] : -INFINITY;
                mx = fmax(mx, x[j]);
            }
#pragma unroll
            for (int off = 16; off; off >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, off));
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < 10; j++) { x[j] = (lane + 32 * j) < 294 ? exp(x[j] - mx) : 0.0; sum += x[j]; }
#pragma unroll
            for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
#pragma unroll
            for (int j = 0; j < 10; j++) if (lane + 32 * j < 294) sPr[lane + 32 * j] = x[j] / sum;
        }
        g = load_node_game(tv, leaf);
        u64 mv = 0;
        if (lane < 6) {
            u64 occ_all = g.occ_me | g.occ_op;
            u64 o = 1ULL << ((g.cells_me >> (8 * lane)) & 0xFF);
            u64 occ = occ_all & ~o, empty = ~occ & CCX_VALID;
            u64 todo = o, reach = 0;
            while (todo) {
                int i = 63 - __clzll((long long)todo);
                todo ^= 1ULL << i;
                u64 nw = expand_cell(i, occ, sT) & ~(reach | o);
                reach |= nw; todo |= nw;
            }
            mv = (neighbours(o) & empty) | reach;
        }
#pragma unroll
        for (int k = 0; k < 6; k++) { dest[k] = shfl64(mv, k); pre[k + 1] = pre[k] + __popcll(dest[k]); }
    }
    if (lane == 0 && w < CCX_MAX_LEAVES) s_cnt[w] = mine ? pre[6] : 0;
    __syncthreads();
    // (2) edge ranges in slot order; an edge pool too small for the round flags the tree (no expansion at all)
    if (threadIdx.x == 0) {
        int ov = ov0, eb = tv.meta[META_NEDGES];
        for (int k = 0; k < m; k++) { s_off[k] = eb; eb += s_cnt[k]; }
        if (!ov && eb > tv.ept) { ov = 1; tv.meta[META_OVERFLOW] = 1; }
        if (!ov) tv.meta[META_NEDGES] = eb;
        s_ov = ov;
    }
    __syncthreads();
    const int ov = s_ov;
    if (mine && !ov) {
        const int eb = s_off[w], total = pre[6];
        const double *p = NET ? sPr : (const double *)pv + slot * CCX_NUM_ACTIONS;
        for (int j = lane; j < total; j += 32) {
            int k = 0;
#pragma unroll
            for (int q = 1; q < 6; q++) k += (j >= pre[q]);
            u64 mk = 0; int base = 0;
#pragma unroll
            for (int q = 0; q < 6; q++) if (k == q) { mk = dest[q]; base = pre[q]; }
            int to = select64(mk, (u32)(j - base));
            int idx = k * 49 + (to >> 3) * 7 + (to & 7);
            tv.eN[eb + j] = 0; tv.eW[eb + j] = 0.0; tv.eQ[eb + j] = 0.0; tv.eP[eb + j] = p[idx];
            tv.eChild[eb + j] = -1;
            tv.eMove[eb + j] = (uint16_t)((k << 8) | to);
        }
        if (lane == 0) {                                         // (leaf record re-read: keeps the registers free across the loop)
            const int32_t *r = lv.rec + 4 * w;
            const u64 info = make_info((u32)eb, (u32)total, 0, 1);
            tv.node[(int64_t)r[0] * NODE_WORDS + 5] = info;
            if (r[1] > 0) tv.eInfo[lv.path[w * lv.path_max + r[1] - 1]] = info;
        }
    }
    __syncthreads();
    // (3) backups in slot order: one virtual loss off every pending path, the real update unless the tree is flagged
    if (w == 0) {
        for (int k = 0; k < m; k++) {
            const int32_t *r = lv.rec + 4 * k;
            const int kk = r[2];
            if (kk != LK_FIRST && kk != LK_DUP) continue;
            const int path_len = r[1];
            const int64_t src = tree * L + (kk == LK_DUP ? r[3] : k);
            const double v = NET && SYM != SYM_OFF ? sym_value<SYM>((const float *)vv + src * SymRows<SYM>::value)
                           : NET ? (double)((const float *)vv)[src] : ((const double *)vv)[src];
            const int32_t *path = lv.path + k * lv.path_max;
            for (int d = lane; d < path_len; d += 32) {
                int e = path[d];
                lv.vl[e] -= 1;
                if (!ov) {
                    bool same = ((path_len - d) & 1) == 0;
                    double delta = __dmul_rn(v, same ? 1.0 : -1.0);
                    u32 N = tv.eN[e] + 1;
                    double W = __dadd_rn(tv.eW[e], delta);
                    tv.eN[e] = N;
                    tv.eW[e] = W;
                    tv.eQ[e] = __ddiv_rn(W, (double)N);
                }
            }
            __syncwarp();
        }
        if (noise && !ov && m > 0 && lv.rec[2] == LK_FIRST && lv.rec[0] == 0) mix_root_noise(tv, lane, noise, noise_normalize != 0);
    }
}

template <bool TIES, bool ENCODE>
__global__ void __launch_bounds__(32 * CCX_MAX_LEAVES)
k_mcts_select_leaves(ccx_trees trees, ccx_leaf_pool lp, int64_t tree0, int L, double cpuct, int budget, uint8_t *__restrict__ planes,
                     u64 *__restrict__ leaf_state, int64_t n_slots)
{
    extern __shared__ __align__(16) uint8_t s_dyn[];       // ENCODE: [L][352] staging of the planes
    const int64_t tree = tree0 + blockIdx.x;
    TreeView tv = tree_view(trees, tree);
    leaves_select<TIES, ENCODE>(tv, leaf_view(trees, lp, tree), tree, L, cpuct, budget, planes, leaf_state, n_slots,
                                s_dyn + (threadIdx.x >> 5) * 352);
}

// expand + backup with the caller's priors p[slot][294] and values v[slot] (float64)
__global__ void __launch_bounds__(32 * CCX_MAX_LEAVES)
k_mcts_backup_leaves(ccx_trees trees, ccx_leaf_pool lp, int64_t tree0, int L, const double *p, const double *v, const double *noise,
                     int noise_stride, int noise_normalize, const uint8_t *__restrict__ jt)
{
    const int64_t tree = tree0 + blockIdx.x;
    TreeView tv = tree_view(trees, tree);
    leaves_backup<false>(tv, leaf_view(trees, lp, tree), tree, L, p, v, noise ? noise + tree * noise_stride : nullptr, noise_normalize,
                         nullptr, jt);
}

// steady state of ccx_mcts_run_net_leaves: finish the previous round (softmax + expand + backup), then select and encode;
// budget 0 in the last launch (nothing left to select: every slot gets the start position, which nobody reads)
template <bool TIES>
__global__ void __launch_bounds__(32 * CCX_MAX_LEAVES)
k_mcts_round_leaves(ccx_trees trees, ccx_leaf_pool lp, int64_t tree0, int L, double cpuct, const float *__restrict__ logits,
                    const float *__restrict__ value, const double *noise, int noise_stride, int noise_normalize,
                    uint8_t *__restrict__ planes, const uint8_t *__restrict__ jt, int budget)
{
    extern __shared__ __align__(16) uint8_t s_dyn[];       // [L][296] float64 priors, then [L][352] staging of the planes
    const int64_t tree = tree0 + blockIdx.x;
    TreeView tv = tree_view(trees, tree);
    const LeafView lv = leaf_view(trees, lp, tree);
    const int w = threadIdx.x >> 5;
    leaves_backup<true>(tv, lv, tree, L, logits, value, noise ? noise + tree * noise_stride : nullptr, noise_normalize,
                        reinterpret_cast<double *>(s_dyn) + w * 296, jt);
    __syncthreads();
    leaves_select<TIES, true>(tv, lv, tree, L, cpuct, budget, planes, nullptr, 0, s_dyn + L * 296 * 8 + w * 352);
}

// the two fused launches above with a mirror-symmetric net evaluation (ccx_net_set_symmetry): slot s owns net rows
// [s * SymRows, (s + 1) * SymRows)
template <bool TIES, int SYM>
__global__ void __launch_bounds__(32 * CCX_MAX_LEAVES)
k_mcts_select_leaves_sym(ccx_trees trees, ccx_leaf_pool lp, int64_t tree0, int L, double cpuct, int budget, uint8_t *__restrict__ planes,
                         u32 k0, u32 k1)
{
    extern __shared__ __align__(16) uint8_t s_dyn[];       // [L][352] staging of the planes
    const int64_t tree = tree0 + blockIdx.x;
    TreeView tv = tree_view(trees, tree);
    leaves_select<TIES, true, SYM>(tv, leaf_view(trees, lp, tree), tree, L, cpuct, budget, planes, nullptr, 0,
                                   s_dyn + (threadIdx.x >> 5) * 352, k0, k1);
}

template <bool TIES, int SYM>
__global__ void __launch_bounds__(32 * CCX_MAX_LEAVES)
k_mcts_round_leaves_sym(ccx_trees trees, ccx_leaf_pool lp, int64_t tree0, int L, double cpuct, const float *__restrict__ logits,
                        const float *__restrict__ value, const double *noise, int noise_stride, int noise_normalize,
                        uint8_t *__restrict__ planes, const uint8_t *__restrict__ jt, int budget, u32 k0, u32 k1)
{
    extern __shared__ __align__(16) uint8_t s_dyn[];       // [L][296] float64 priors, then [L][352] staging of the planes
    const int64_t tree = tree0 + blockIdx.x;
    TreeView tv = tree_view(trees, tree);
    const LeafView lv = leaf_view(trees, lp, tree);
    const int w = threadIdx.x >> 5;
    leaves_backup<true, SYM>(tv, lv, tree, L, logits, value, noise ? noise + tree * noise_stride : nullptr, noise_normalize,
                             reinterpret_cast<double *>(s_dyn) + w * 296, jt, k0, k1);
    __syncthreads();
    leaves_select<TIES, true, SYM>(tv, lv, tree, L, cpuct, budget, planes, nullptr, 0, s_dyn + L * 296 * 8 + w * 352, k0, k1);
}

__global__ void k_mcts_leaf_budget(ccx_leaf_pool lp, int64_t n, int sims)
{
    int64_t tree = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tree < n) lp.meta[tree * 2 + 1] = sims;
}

// ---- finalize (MCTS.py:131-137): visit counts, pi = N^(1/tau) / sum, root Q ---------------------------
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_finalize(ccx_trees trees, int64_t n, double inv_tau, u32 *__restrict__ visits, double *__restrict__ pi,
                double *__restrict__ q, int32_t *__restrict__ n_nodes)
{
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    for (int a = lane; a < CCX_NUM_ACTIONS; a += 32) {
        visits[tree * CCX_NUM_ACTIONS + a] = 0;
        if (pi) pi[tree * CCX_NUM_ACTIONS + a] = 0.0;
        if (q) q[tree * CCX_NUM_ACTIONS + a] = 0.0;
    }
    __syncwarp();
    u64 info = tv.node[5];
    int ne = info_ne(info), eb = info_eb(info);
    double sum = 0.0;
    for (int j = lane; j < ne; j += 32) {
        u32 N = tv.eN[eb + j];
        double pw = inv_tau == 1.0 ? (double)N : pow((double)N, inv_tau);       // MCTS.py:132
        sum += pw;
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);   // exact for tau = 1 (integers)
    for (int j = lane; j < ne; j += 32) {
        u32 N = tv.eN[eb + j];
        u32 mv = tv.eMove[eb + j];
        int to = (int)(mv & 0xFF);
        int idx = (int)(mv >> 8) * 49 + (to >> 3) * 7 + (to & 7);
        visits[tree * CCX_NUM_ACTIONS + idx] = N;
        if (pi) {
            double pw = inv_tau == 1.0 ? (double)N : pow((double)N, inv_tau);
            pi[tree * CCX_NUM_ACTIONS + idx] = sum > 0.0 ? __ddiv_rn(pw, sum) : 0.0;       // MCTS.py:137
        }
        if (q) q[tree * CCX_NUM_ACTIONS + idx] = N ? __ddiv_rn(tv.eW[eb + j], (double)N) : 0.0;
    }
    if (n_nodes && lane == 0)
        n_nodes[tree] = tv.meta[META_OVERFLOW] ? -tv.meta[META_OVERFLOW] : tv.meta[META_NEDGES] + 1;   // reference node count: root + one per edge
}

// ---- Gumbel search (ccx_mcts_set_gumbel; mctx gumbel_muzero_policy with qtransform_completed_by_mix_value) ------------
// Own kernels beside the PUCT ones (which stay as they are): one leaf per round, the root chosen by sequential halving
// over Gumbel-perturbed logits, interior nodes by argmax of pi' - N / (1 + sum N), pi' = softmax(logit + sigma(q^)).
// Fixed arithmetic, restated literally by the CPU test restatement:
//   * log / exp are ccx_fpmath.cuh's; every operation is an explicit round-to-nearest one, evaluated left to right;
//   * every float64 sum is a per-lane sequential sum over chunks c = 0..3 (edge j = lane + 32c, 0.0 past the last edge)
//     followed by an xor butterfly over offsets 16, 8, 4, 2, 1; maxima and minima are order-free;
//   * arg-maxes take the first maximal edge (no tie rule).
#define GUMBEL_EDGES 128            // root Gumbel draws per tree (a node has at most 126 legal moves)
struct ccx_gumbel_dev {             // by-value kernel argument (part of the cached round graph's key)
    double *vraw = nullptr;         // [T][NPT] evaluator value of every expanded node, in the sign of the Q of its edges
    double *g = nullptr;            // [T][GUMBEL_EDGES] Gumbel draws of the root edges (scale included)
    int32_t *mp = nullptr;          // [T] considered count m' = min(m, root edges)
    const int32_t *table = nullptr; // [rows][cols] considered visits at root simulation k (ccx_gumbel_table.h)
    int32_t rows = 0, cols = 0, npt = 0, m = 0;
    double scale = 1.0, c_visit = 50.0, c_scale = 0.1;
    u32 seed_lo = 0, seed_hi = 0;
};

__device__ __forceinline__ double warp_sum_f64(double s)
{
#pragma unroll
    for (int off = 16; off; off >>= 1) s = __dadd_rn(s, __shfl_xor_sync(FULL, s, off));
    return s;
}
__device__ __forceinline__ double warp_max_f64(double s)
{
#pragma unroll
    for (int off = 16; off; off >>= 1) s = fmax(s, __shfl_xor_sync(FULL, s, off));
    return s;
}
__device__ __forceinline__ double warp_min_f64(double s)
{
#pragma unroll
    for (int off = 16; off; off >>= 1) s = fmin(s, __shfl_xor_sync(FULL, s, off));
    return s;
}

// the edge statistics of one node turned into logits and sigma(q^) (completed Q by the mixed value, rescaled by the node's
// min / max, times (c_visit + max N) c_scale); lanes hold edges lane + 32c
struct GumbelNode { double logit[4], sigma[4], maxlogit; u32 nsum, nmax; };

__device__ __forceinline__ void gumbel_node(int lane, int ne, const u32 *N, const double *Q, const double *P, double vraw,
                                            const ccx_gumbel_dev &gd, GumbelNode &o)
{
    double mx = -INFINITY;
    u32 nsum = 0, nmax = 0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const bool in = lane + 32 * c < ne;
        o.logit[c] = in ? fm_log(P[c] > DBL_MIN ? P[c] : DBL_MIN) : -INFINITY;
        mx = fmax(mx, o.logit[c]);
        nsum += N[c];
        nmax = max(nmax, N[c]);
    }
    mx = warp_max_f64(mx);
    o.maxlogit = mx;
    o.nsum = __reduce_add_sync(FULL, nsum);
    o.nmax = __reduce_max_sync(FULL, nmax);
    double e[4], z = 0.0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        e[c] = lane + 32 * c < ne ? fm_exp(__dsub_rn(o.logit[c], mx)) : 0.0;
        z = __dadd_rn(z, e[c]);
    }
    z = warp_sum_f64(z);
    double sp = 0.0, spq = 0.0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const bool vis = lane + 32 * c < ne && N[c] > 0;
        double pt = __ddiv_rn(e[c], z);
        pt = pt > DBL_MIN ? pt : DBL_MIN;                        // mctx: prior probabilities floored at the smallest normal
        sp = __dadd_rn(sp, vis ? pt : 0.0);
        spq = __dadd_rn(spq, vis ? __dmul_rn(pt, Q[c]) : 0.0);
    }
    sp = warp_sum_f64(sp);
    spq = warp_sum_f64(spq);
    const double ns = (double)o.nsum;
    const double vmix = o.nsum ? __ddiv_rn(__dadd_rn(vraw, __ddiv_rn(__dmul_rn(ns, spq), sp)), __dadd_rn(1.0, ns)) : vraw;
    double q[4], qmin = INFINITY, qmax = -INFINITY;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        q[c] = N[c] > 0 ? Q[c] : vmix;
        if (lane + 32 * c < ne) { qmin = fmin(qmin, q[c]); qmax = fmax(qmax, q[c]); }
    }
    qmin = warp_min_f64(qmin);
    qmax = warp_max_f64(qmax);
    double den = __dsub_rn(qmax, qmin);
    den = den > 1e-8 ? den : 1e-8;
    const double vs = __dmul_rn(__dadd_rn(gd.c_visit, (double)o.nmax), gd.c_scale);
#pragma unroll
    for (int c = 0; c < 4; c++)
        o.sigma[c] = lane + 32 * c < ne ? __dmul_rn(vs, __ddiv_rn(__dsub_rn(q[c], qmin), den)) : 0.0;
}

// pi'(a) = softmax(logit + sigma) over the node's edges (w[c] / W)
__device__ __forceinline__ double gumbel_improved(int lane, int ne, const GumbelNode &o, double *w)
{
    double zz[4], zmax = -INFINITY;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        zz[c] = lane + 32 * c < ne ? __dadd_rn(o.logit[c], o.sigma[c]) : -INFINITY;
        zmax = fmax(zmax, zz[c]);
    }
    zmax = warp_max_f64(zmax);
    double W = 0.0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        w[c] = lane + 32 * c < ne ? fm_exp(__dsub_rn(zz[c], zmax)) : 0.0;
        W = __dadd_rn(W, w[c]);
    }
    return warp_sum_f64(W);
}

// root score of mctx's score_considered: max(-1e9, g + (logit - max logit) + sigma) on the edges with N == considered visit
__device__ __forceinline__ double gumbel_root_score(const GumbelNode &o, int c, double g, u32 N, u32 cv)
{
    return N == cv ? fmax(-1e9, __dadd_rn(__dadd_rn(g, __dsub_rn(o.logit[c], o.maxlogit)), o.sigma[c])) : -INFINITY;
}

// first maximal edge over the warp (edge 0 when no score is above -inf)
__device__ __forceinline__ int warp_argmax_first(double best, int besti)
{
    const u64 u = (u64)__double_as_longlong(best + 0.0);
    const u64 key = (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
    const u32 hi = (u32)(key >> 32), lo = (u32)key;
    const u32 mhi = __reduce_max_sync(FULL, hi);
    const u32 mlo = __reduce_max_sync(FULL, hi == mhi ? lo : 0u);
    const u32 b = __reduce_min_sync(FULL, (hi == mhi && lo == mlo) ? (u32)besti : 0x7FFFFFFFu);
    return b == 0x7FFFFFFFu ? 0 : (int)b;
}

// one descent under the Gumbel rules (the one-leaf select_leaf with the edge statistics prefetched)
__device__ __forceinline__ int gumbel_select_leaf(const TreeView &tv, const ccx_gumbel_dev &gd, int lane, int &path_len, int &leaf_kind)
{
    int node = 0, depth = 0;
    u64 info = tv.node[5];
    const int64_t tree = (int64_t)tv.tree_index;
    for (;;) {
        const int ne = info_ne(info);
        if (info_winner(info)) { leaf_kind = LEAF_TERMINAL; break; }
        if (ne == 0) { leaf_kind = LEAF_EVAL; break; }
        const int eb = info_eb(info);
        u32 Nr[4]; double Qr[4], Pr[4]; int Cr[4]; u64 Ir[4];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int j = lane + 32 * c;
            const bool in = j < ne;
            Cr[c] = in ? tv.eChild[eb + j] : -1;
            Ir[c] = in ? tv.eInfo[eb + j] : 0ULL;
            Nr[c] = in ? tv.eN[eb + j] : 0u;
            Qr[c] = in ? tv.eQ[eb + j] : 0.0;
            Pr[c] = in ? tv.eP[eb + j] : 0.0;
        }
        GumbelNode o;
        gumbel_node(lane, ne, Nr, Qr, Pr, gd.vraw[tree * gd.npt + node], gd, o);
        double best = -INFINITY; int besti = 0x7FFFFFFF;
        if (node == 0) {                                          // root: sequential halving
            const int k = min((int)o.nsum, gd.cols - 1);
            const u32 cv = (u32)gd.table[gd.mp[tree] * gd.cols + k];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int j = lane + 32 * c;
                if (j < ne) {
                    const double s = gumbel_root_score(o, c, gd.g[tree * GUMBEL_EDGES + j], Nr[c], cv);
                    if (s > best) { best = s; besti = j; }
                }
            }
        } else {                                                  // interior: pi' - N / (1 + sum N)
            double w[4];
            const double W = gumbel_improved(lane, ne, o, w);
            const double d = __dadd_rn(1.0, (double)o.nsum);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int j = lane + 32 * c;
                if (j < ne) {
                    const double s = __dsub_rn(__ddiv_rn(w[c], W), __ddiv_rn((double)Nr[c], d));
                    if (s > best) { best = s; besti = j; }
                }
            }
        }
        besti = warp_argmax_first(best, besti);
        const int e = eb + besti;
        if (lane == 0 && depth < tv.path_max) tv.path[depth] = e;
        depth++;
        const int chunk = besti >> 5, src = besti & 31;
        const int child = __shfl_sync(FULL, chunk == 0 ? Cr[0] : chunk == 1 ? Cr[1] : chunk == 2 ? Cr[2] : Cr[3], src);
        const u64 cinfo = shfl64(chunk == 0 ? Ir[0] : chunk == 1 ? Ir[1] : chunk == 2 ? Ir[2] : Ir[3], src);
        if (child < 0) {                                          // first visit: materialise the child (as select_leaf)
            const int nn = tv.meta[META_NNODES];
            if (nn >= tv.npt) { if (lane == 0) tv.meta[META_OVERFLOW] = 1; leaf_kind = LEAF_DEAD; node = 0; break; }
            Game g = load_node_game(tv, node);
            const u32 mv = tv.eMove[e];
            const int id = (int)(mv >> 8), to = (int)(mv & 0xFF);
            apply_move(g, id, (int)((g.cells_me >> (8 * id)) & 0xFF), to);
            const int w = winner_of(g);
            __syncwarp();
            if (lane == 0) {
                store_node(tv, nn, g, make_info(0, 0, (u32)w, 0));
                tv.eChild[e] = nn;
                tv.eInfo[e] = make_info(0, 0, (u32)w, 0);
                tv.meta[META_NNODES] = nn + 1;
            }
            __syncwarp();
            node = nn;
            leaf_kind = w ? LEAF_TERMINAL : LEAF_EVAL;
            break;
        }
        node = child;
        info = cinfo;
    }
    path_len = depth;
    return node;
}

// after an expansion: the node's value; at the root also the Gumbel draws (Philox4x32-10, key (seed lo, uid lo), counter
// (search serial, edge, uid hi, seed hi), 64 bits y:x -> fm_gumbel, times scale) and m'
__device__ __forceinline__ void gumbel_after_expand(const TreeView &tv, const ccx_gumbel_dev &gd, int lane, int leaf, double v)
{
    const int64_t tree = (int64_t)tv.tree_index;
    if (lane == 0) gd.vraw[tree * gd.npt + leaf] = v;
    if (leaf != 0) return;
    const int ne = info_ne(tv.node[5]);
    const u64 uid = tv.tie_uids ? (u64)tv.tie_uids[tree] : (((u64)tv.tie[3] << 32) | tv.tie[2]) + (u64)tree;
    const u32 serial = (u32)tv.meta[META_SERIAL];
    for (int j = lane; j < ne; j += 32) {
        const Philox4 r = philox4x32_10(gd.seed_lo, (u32)uid, serial, (u32)j, (u32)(uid >> 32), gd.seed_hi);
        gd.g[tree * GUMBEL_EDGES + j] = __dmul_rn(gd.scale, fm_gumbel(((u64)r.y << 32) | r.x));
    }
    if (lane == 0) gd.mp[tree] = min(gd.m, ne);
}

__device__ __forceinline__ void gumbel_select_phase(const TreeView &tv, const ccx_gumbel_dev &gd, int lane, int &leaf, int &kind)
{
    if (tv.meta[META_OVERFLOW]) {
        if (lane == 0) tv.meta[META_LEAFKIND] = LEAF_DEAD;
        kind = LEAF_DEAD; leaf = 0;
        return;
    }
    int path_len;
    leaf = gumbel_select_leaf(tv, gd, lane, path_len, kind);
    __syncwarp();
    if (kind == LEAF_TERMINAL) backup(tv, lane, path_len, 0.0, true);
    if (lane == 0) { tv.meta[META_PATHLEN] = path_len; tv.meta[META_LEAF] = leaf; tv.meta[META_LEAFKIND] = kind; }
}

// round trip, phase A (ccx_mcts_select in the Gumbel mode)
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_select_gumbel(ccx_trees trees, ccx_gumbel_dev gd, int64_t n, u64 *__restrict__ leaf_state)
{
    const int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    int leaf, kind;
    gumbel_select_phase(tv, gd, lane, leaf, kind);
    if (lane < 5) {
        const u64 dummy = lane == 0 ? CCX_START_OCC1 : lane == 1 ? CCX_START_OCC2 : lane == 2 ? CCX_START_CELLS1
                        : lane == 3 ? CCX_START_CELLS2 : CCX_START_META;
        leaf_state[lane * n + tree] = kind == LEAF_DEAD ? dummy : tv.node[(int64_t)leaf * NODE_WORDS + lane];
    }
}

// round trip, phase B (ccx_mcts_expand_backup in the Gumbel mode): priors p[n][294], values v[n] in float64
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_expand_backup_gumbel(ccx_trees trees, ccx_gumbel_dev gd, int64_t n, const double *__restrict__ p, const double *__restrict__ v,
                            const uint8_t *__restrict__ jt)
{
    const int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    if (tv.meta[META_LEAFKIND] != LEAF_EVAL) return;
    const int leaf = tv.meta[META_LEAF], path_len = tv.meta[META_PATHLEN];
    const Game g = load_node_game(tv, leaf);
    const TablePrior pr = {p + tree * CCX_NUM_ACTIONS};
    if (expand_node(tv, lane, leaf, g, pr, jt, path_len > 0 ? tv.path[path_len - 1] : -1)) {
        backup(tv, lane, path_len, v[tree], false);
        gumbel_after_expand(tv, gd, lane, leaf, v[tree]);
    }
}

// fused net loop: do_softmax_expand_backup (without root noise), then the node's value and the root's draws
template <int SYM = SYM_OFF>
__device__ __forceinline__ void gumbel_softmax_expand_backup(const TreeView &tv, const ccx_gumbel_dev &gd, int lane,
                                                             const float *__restrict__ lg, double v, double *__restrict__ pr,
                                                             const uint8_t *__restrict__ sT, u32 k0 = 0, u32 k1 = 0)
{
    if (tv.meta[META_LEAFKIND] != LEAF_EVAL) return;
    do_softmax_expand_backup<SYM>(tv, lane, lg, v, nullptr, 0, pr, sT, k0, k1);
    __syncwarp();
    if (!tv.meta[META_OVERFLOW]) gumbel_after_expand(tv, gd, lane, tv.meta[META_LEAF], v);
}

template <int SYM = SYM_OFF>
__device__ __forceinline__ void gumbel_select_encode(const TreeView &tv, const ccx_gumbel_dev &gd, int lane, uint8_t *__restrict__ sp,
                                                     uint8_t *__restrict__ dst, u32 k0 = 0, u32 k1 = 0)
{
    int leaf, kind;
    gumbel_select_phase(tv, gd, lane, leaf, kind);
    Game g;
    if (kind == LEAF_DEAD) reset_start(g);
    else g = load_node_game(tv, leaf);
    if (SYM != SYM_OFF) sym_encode<SYM>(g, lane, k0, k1, sp, dst);
    else encode_planes(g, lane, sp, dst);
}

// the fused net loop's three launches (as k_mcts_select_encode, k_mcts_round, k_mcts_softmax_expand_backup)
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_select_encode_gumbel(ccx_trees trees, ccx_gumbel_dev gd, int64_t tree0, int64_t n, uint8_t *__restrict__ planes)
{
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    const int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    gumbel_select_encode(tv, gd, threadIdx.x & 31, sP[threadIdx.x >> 5], planes + tree * 343);
}

__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_round_gumbel(ccx_trees trees, ccx_gumbel_dev gd, int64_t tree0, int64_t n, const float *__restrict__ logits,
                    const float *__restrict__ value, uint8_t *__restrict__ planes, const uint8_t *__restrict__ jt)
{
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    const int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    gumbel_softmax_expand_backup(tv, gd, lane, logits + tree * 294, (double)value[tree], sPr[threadIdx.x >> 5], jt);
    __syncwarp();
    __threadfence_block();
    gumbel_select_encode(tv, gd, lane, sP[threadIdx.x >> 5], planes + tree * 343);
}

__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_softmax_expand_backup_gumbel(ccx_trees trees, ccx_gumbel_dev gd, int64_t tree0, int64_t n, const float *__restrict__ logits,
                                    const float *__restrict__ value, const uint8_t *__restrict__ jt)
{
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    const int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    gumbel_softmax_expand_backup(tv, gd, threadIdx.x & 31, logits + tree * 294, (double)value[tree], sPr[threadIdx.x >> 5], jt);
}

// the three launches above with a mirror-symmetric net evaluation (ccx_net_set_symmetry), rows as k_mcts_round_sym
template <int SYM>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_select_encode_gumbel_sym(ccx_trees trees, ccx_gumbel_dev gd, int64_t tree0, int64_t n, uint8_t *__restrict__ planes, u32 k0, u32 k1)
{
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    const int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    gumbel_select_encode<SYM>(tv, gd, threadIdx.x & 31, sP[threadIdx.x >> 5], planes + tree * SymRows<SYM>::value * 343, k0, k1);
}

template <int SYM>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK, 14)
k_mcts_round_gumbel_sym(ccx_trees trees, ccx_gumbel_dev gd, int64_t tree0, int64_t n, const float *__restrict__ logits,
                        const float *__restrict__ value, uint8_t *__restrict__ planes, const uint8_t *__restrict__ jt, u32 k0, u32 k1)
{
    constexpr int R = SymRows<SYM>::value;
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    __shared__ __align__(16) uint8_t sP[MCTS_WARPS_PER_BLOCK][352];
    const int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    gumbel_softmax_expand_backup<SYM>(tv, gd, lane, logits + tree * R * 294, sym_value<SYM>(value + tree * R), sPr[threadIdx.x >> 5], jt,
                                      k0, k1);
    __syncwarp();
    __threadfence_block();
    gumbel_select_encode<SYM>(tv, gd, lane, sP[threadIdx.x >> 5], planes + tree * R * 343, k0, k1);
}

template <int SYM>
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_softmax_expand_backup_gumbel_sym(ccx_trees trees, ccx_gumbel_dev gd, int64_t tree0, int64_t n, const float *__restrict__ logits,
                                        const float *__restrict__ value, const uint8_t *__restrict__ jt, u32 k0, u32 k1)
{
    constexpr int R = SymRows<SYM>::value;
    __shared__ double sPr[MCTS_WARPS_PER_BLOCK][296];
    const int64_t tree = tree0 + (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (tree >= tree0 + n) return;
    TreeView tv = tree_view(trees, tree);
    gumbel_softmax_expand_backup<SYM>(tv, gd, threadIdx.x & 31, logits + tree * R * 294, sym_value<SYM>(value + tree * R),
                                      sPr[threadIdx.x >> 5], jt, k0, k1);
}

// result of a Gumbel search: visits, Q and node counts as k_mcts_finalize; action = the root score's arg-max with considered
// visit max N (-1 for an inactive, overflowed or unexpanded root); pi = softmax(logit + sigma) over the root's edges
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_finalize_gumbel(ccx_trees trees, ccx_gumbel_dev gd, int64_t n, u32 *__restrict__ visits, double *__restrict__ pi,
                       double *__restrict__ q, int32_t *__restrict__ action, int32_t *__restrict__ n_nodes)
{
    const int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    for (int a = lane; a < CCX_NUM_ACTIONS; a += 32) {
        visits[tree * CCX_NUM_ACTIONS + a] = 0;
        if (pi) pi[tree * CCX_NUM_ACTIONS + a] = 0.0;
        if (q) q[tree * CCX_NUM_ACTIONS + a] = 0.0;
    }
    __syncwarp();
    const u64 info = tv.node[5];
    const int ne = info_ne(info), eb = info_eb(info);
    const int ov = tv.meta[META_OVERFLOW];
    u32 Nr[4]; double Qr[4], Pr[4]; int idx[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const int j = lane + 32 * c;
        const bool in = j < ne;
        Nr[c] = in ? tv.eN[eb + j] : 0u;
        Qr[c] = in ? tv.eQ[eb + j] : 0.0;
        Pr[c] = in ? tv.eP[eb + j] : 0.0;
        idx[c] = 0;
        if (in) {
            const u32 mv = tv.eMove[eb + j];
            const int to = (int)(mv & 0xFF);
            idx[c] = (int)(mv >> 8) * 49 + (to >> 3) * 7 + (to & 7);
            visits[tree * CCX_NUM_ACTIONS + idx[c]] = Nr[c];
            if (q) q[tree * CCX_NUM_ACTIONS + idx[c]] = Nr[c] ? __ddiv_rn(tv.eW[eb + j], (double)Nr[c]) : 0.0;
        }
    }
    int act = -1;
    if (!ov && ne > 0) {
        GumbelNode o;
        gumbel_node(lane, ne, Nr, Qr, Pr, gd.vraw[tree * gd.npt], gd, o);
        double w[4];
        const double W = gumbel_improved(lane, ne, o, w);
        double best = -INFINITY; int besti = 0x7FFFFFFF;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int j = lane + 32 * c;
            if (j < ne) {
                if (pi) pi[tree * CCX_NUM_ACTIONS + idx[c]] = __ddiv_rn(w[c], W);
                const double s = gumbel_root_score(o, c, gd.g[tree * GUMBEL_EDGES + j], Nr[c], o.nmax);
                if (s > best) { best = s; besti = j; }
            }
        }
        besti = warp_argmax_first(best, besti);
        const int chunk = besti >> 5;
        act = __shfl_sync(FULL, chunk == 0 ? idx[0] : chunk == 1 ? idx[1] : chunk == 2 ? idx[2] : idx[3], besti & 31);
    }
    if (lane == 0) {
        if (action) action[tree] = act;
        if (n_nodes) n_nodes[tree] = ov ? -ov : tv.meta[META_NEDGES] + 1;
    }
}

// ---- root edge access for the Python Node/Edge mirror (MCTS.py:24-37; selfplay.py:121-124 mutates P) ----
__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_get_root(ccx_trees trees, int64_t n, int stride, int32_t *__restrict__ n_edges, uint16_t *__restrict__ moves,
                u32 *__restrict__ N, double *__restrict__ W, double *__restrict__ P)
{
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    u64 info = tv.node[5];
    int ne = info_ne(info), eb = info_eb(info);
    if (lane == 0) n_edges[tree] = ne;
    for (int j = lane; j < ne && j < stride; j += 32) {
        moves[tree * stride + j] = tv.eMove[eb + j];
        N[tree * stride + j] = tv.eN[eb + j];
        W[tree * stride + j] = tv.eW[eb + j];
        P[tree * stride + j] = tv.eP[eb + j];
    }
}

__global__ void __launch_bounds__(32 * MCTS_WARPS_PER_BLOCK)
k_mcts_set_root_priors(ccx_trees trees, int64_t n, int stride, const double *__restrict__ P)
{
    int64_t tree = (int64_t)blockIdx.x * MCTS_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (tree >= n) return;
    TreeView tv = tree_view(trees, tree);
    u64 info = tv.node[5];
    int ne = info_ne(info), eb = info_eb(info);
    for (int j = lane; j < ne && j < stride; j += 32) tv.eP[eb + j] = P[tree * stride + j];
}

// ---- host side ----------------------------------------------------------------------------------------

// cached CUDA graph of the round loop (see ccx_mcts_run_net)
struct ccx_round_graph {
    cudaGraphExec_t exec = nullptr;
    bool seen = false;
    uint64_t epoch = 0;
    int64_t n = 0, launches = 0;
    int32_t rounds = 0, stride = 0, normalize = 0;
    int32_t leaves = 1;         // leaf-parallel rounds (ccx_mcts_run_net_leaves): leaves > 1, `rounds` = selections of the call
    double cpuct = 0.0;
    const double *noise = nullptr;
    ccx_trees trees;
    ccx_leaf_pool pool;
    int32_t gumbel = 0;         // Gumbel mode: its device state (buffers and parameters) is part of the key
    ccx_gumbel_dev gdev;
};

void ccx_round_graph_free(ccx_handle *h)
{
    ccx_round_graph *g = (ccx_round_graph *)h->round_graph;
    if (g) {
        if (g->exec) cudaGraphExecDestroy(g->exec);
        delete g;
    }
    h->round_graph = nullptr;
    if (h->cap_stream) { cudaStreamDestroy(h->cap_stream); h->cap_stream = nullptr; }
}

void ccx_trees_set_uids(ccx_handle *h, const int64_t *uids)
{
    if (h->trees) h->trees->tie_uids = uids;          // by-value kernel argument: part of the cached round graph's key
}

static void leaf_pool_free(ccx_handle *h)
{
    ccx_leaf_pool *lp = (ccx_leaf_pool *)h->leaf_pool;
    if (!lp) return;
    void *ptrs[] = {lp->path, lp->rec, lp->meta, lp->vl};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete lp;
    h->leaf_pool = nullptr;
}

// scratch of the tree-reuse gather: a node / edge pool per tree sized for the largest subtree a reuse begin may carry (no
// paths, no per-tree meta), the BFS queue's source indices and the per-tree match records
struct ccx_reuse_pool {
    ccx_trees scratch;
    int32_t *qsrc = nullptr;    // [T][scratch NPT]
    int32_t *rec = nullptr;     // [T][4]
    size_t bytes = 0;
};

static void reuse_pool_free(ccx_handle *h)
{
    ccx_reuse_pool *rp = (ccx_reuse_pool *)h->reuse_pool;
    if (!rp) return;
    const ccx_trees &t = rp->scratch;
    void *ptrs[] = {t.node, t.eN, t.eW, t.eP, t.eQ, t.eChild, t.eInfo, t.eMove, rp->qsrc, rp->rec};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete rp;
    h->reuse_pool = nullptr;
}

// device state of the Gumbel mode for the current trees (ccx_gumbel_dev) and the (m, S) its schedule table was built for
struct ccx_gumbel_pool {
    ccx_gumbel_dev dev;
    int64_t cap_trees = 0;
    int32_t table_m = -1, table_s = -1;
    int32_t *table = nullptr;
    size_t bytes = 0;
};

static void gumbel_pool_free(ccx_handle *h)
{
    ccx_gumbel_pool *gp = (ccx_gumbel_pool *)h->gumbel_pool;
    if (!gp) return;
    void *ptrs[] = {gp->dev.vraw, gp->dev.g, gp->dev.mp, gp->table};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete gp;
    h->gumbel_pool = nullptr;
}

void ccx_trees_free(ccx_handle *h)
{
    leaf_pool_free(h);
    reuse_pool_free(h);
    gumbel_pool_free(h);
    ccx_trees *t = h->trees;
    if (!t) return;
    ccx_round_graph_free(h);
    void *ptrs[] = {t->node, t->eN, t->eW, t->eP, t->eQ, t->eChild, t->eInfo, t->eMove, t->path, t->tree_meta, t->tie_params};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete t;
    h->trees = nullptr;
}

// node / edge / path budgets per tree: one search's (num_itr + 2 nodes, edges_per_tree or 64 (num_itr + 1) edges), times
// 1 + carry for the trees of a reuse begin (ccx_mcts_begin_reuse), so that a carried tree overflows no sooner than a fresh one
static int trees_reserve(ccx_handle *h, int64_t n, int32_t num_itr, int32_t edges_per_tree, int32_t carry = 0)
{
    {   // per device: the constant table lives in this module's image on the handle's device
        static bool filled[64] = {false};
        if (h->device >= 0 && h->device < 64 && !filled[h->device]) {
            static double host_sqrt[SQRT_TABLE];
            for (int i = 0; i < SQRT_TABLE; i++) host_sqrt[i] = sqrt((double)i);
            CCX_CUDA(h, cudaMemcpyToSymbol(c_sqrt, host_sqrt, sizeof(host_sqrt)));
            filled[h->device] = true;
        }
    }
    int32_t npt = (1 + carry) * (num_itr + 2);
    int32_t ept = (1 + carry) * (edges_per_tree > 0 ? edges_per_tree : 64 * (num_itr + 1));
    int32_t pm = (1 + carry) * (num_itr + 2);
    ccx_trees *t = h->trees;
    if (t && t->cap_trees >= n && t->nodes_per_tree >= npt && t->edges_per_tree == ept && t->path_max >= pm) return CCX_OK;
    ccx_trees_free(h);
    h->epoch++;
    h->pool_gen++;
    t = new (std::nothrow) ccx_trees();
    if (!t) return CCX_ERR_NOMEM;
    h->trees = t;
    t->tie_mode = h->tie_mode;
    t->tie_uids = h->slot_ids;
    t->cap_trees = n; t->nodes_per_tree = npt; t->edges_per_tree = ept; t->path_max = pm;
    size_t T = (size_t)n;
    CCX_CUDA(h, cudaMalloc(&t->node, T * npt * NODE_WORDS * 8));
    CCX_CUDA(h, cudaMalloc(&t->eN, T * ept * 4));
    CCX_CUDA(h, cudaMalloc(&t->eW, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&t->eP, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&t->eQ, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&t->eChild, T * ept * 4));
    CCX_CUDA(h, cudaMalloc(&t->eInfo, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&t->eMove, T * ept * 2));
    CCX_CUDA(h, cudaMalloc(&t->path, T * pm * 4));
    CCX_CUDA(h, cudaMalloc(&t->tree_meta, T * 8 * 4));
    CCX_CUDA(h, cudaMalloc(&t->tie_params, 16));
    {
        const u32 tp[4] = {(u32)h->tie_seed, (u32)(h->tie_seed >> 32), (u32)(uint64_t)h->tie_uid0, (u32)((uint64_t)h->tie_uid0 >> 32)};
        CCX_CUDA(h, cudaMemcpyAsync(t->tie_params, tp, 16, cudaMemcpyHostToDevice, h->stream));    // pageable source: staged before the call returns
    }
    t->bytes = T * ((size_t)npt * NODE_WORDS * 8 + (size_t)ept * 42 + (size_t)pm * 4 + 32);
    return CCX_OK;
}

static inline unsigned tree_blocks(int64_t n) { return (unsigned)((n + MCTS_WARPS_PER_BLOCK - 1) / MCTS_WARPS_PER_BLOCK); }

// scratch of the reuse gather for the current trees: npt nodes and ept edges per tree
static int reuse_pool_reserve(ccx_handle *h, int32_t npt, int32_t ept)
{
    const ccx_trees *t = h->trees;
    ccx_reuse_pool *rp = (ccx_reuse_pool *)h->reuse_pool;
    if (rp && rp->scratch.cap_trees >= t->cap_trees && rp->scratch.nodes_per_tree >= npt && rp->scratch.edges_per_tree >= ept)
        return CCX_OK;
    reuse_pool_free(h);
    rp = new (std::nothrow) ccx_reuse_pool();
    if (!rp) return CCX_ERR_NOMEM;
    h->reuse_pool = rp;
    ccx_trees &s = rp->scratch;
    const size_t T = (size_t)t->cap_trees;
    s.cap_trees = t->cap_trees; s.nodes_per_tree = npt; s.edges_per_tree = ept;
    CCX_CUDA(h, cudaMalloc(&s.node, T * npt * NODE_WORDS * 8));
    CCX_CUDA(h, cudaMalloc(&s.eN, T * ept * 4));
    CCX_CUDA(h, cudaMalloc(&s.eW, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&s.eP, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&s.eQ, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&s.eChild, T * ept * 4));
    CCX_CUDA(h, cudaMalloc(&s.eInfo, T * ept * 8));
    CCX_CUDA(h, cudaMalloc(&s.eMove, T * ept * 2));
    CCX_CUDA(h, cudaMalloc(&rp->qsrc, T * npt * 4));
    CCX_CUDA(h, cudaMalloc(&rp->rec, T * 16));
    rp->bytes = T * ((size_t)npt * (NODE_WORDS * 8 + 4) + (size_t)ept * 42 + 16);
    return CCX_OK;
}

// per-leaf storage of the leaf-parallel rounds for the current trees, grown to `leaves` slots per tree; the virtual-loss
// counts start at zero and every backup phase returns them to zero
static int leaf_pool_reserve(ccx_handle *h, int32_t leaves)
{
    ccx_trees *t = h->trees;
    ccx_leaf_pool *lp = (ccx_leaf_pool *)h->leaf_pool;
    if (lp && lp->cap_leaves >= leaves) return CCX_OK;
    leaf_pool_free(h);
    h->epoch++;
    lp = new (std::nothrow) ccx_leaf_pool();
    if (!lp) return CCX_ERR_NOMEM;
    h->leaf_pool = lp;
    const size_t T = (size_t)t->cap_trees;
    lp->cap_leaves = leaves; lp->path_max = t->path_max;
    CCX_CUDA(h, cudaMalloc(&lp->path, T * leaves * t->path_max * 4));
    CCX_CUDA(h, cudaMalloc(&lp->rec, T * leaves * 16));
    CCX_CUDA(h, cudaMalloc(&lp->meta, T * 8));
    CCX_CUDA(h, cudaMalloc(&lp->vl, T * t->edges_per_tree));
    CCX_CUDA(h, cudaMemsetAsync(lp->rec, 0, T * leaves * 16, h->stream));
    CCX_CUDA(h, cudaMemsetAsync(lp->meta, 0, T * 8, h->stream));
    CCX_CUDA(h, cudaMemsetAsync(lp->vl, 0, T * t->edges_per_tree, h->stream));
    lp->bytes = T * ((size_t)leaves * t->path_max * 4 + (size_t)leaves * 16 + 8 + (size_t)t->edges_per_tree);
    return CCX_OK;
}

// Gumbel state for the current trees and a search of S = sims simulations after the root expansion: per-node values and root
// draws sized to the trees, the schedule table rebuilt when (m, S) changes; the parameters are refreshed on every call
static int gumbel_pool_reserve(ccx_handle *h, int32_t sims)
{
    const ccx_trees *t = h->trees;
    ccx_gumbel_pool *gp = (ccx_gumbel_pool *)h->gumbel_pool;
    if (!gp || gp->cap_trees < t->cap_trees || gp->dev.npt != t->nodes_per_tree) {
        gumbel_pool_free(h);
        h->epoch++;
        gp = new (std::nothrow) ccx_gumbel_pool();
        if (!gp) return CCX_ERR_NOMEM;
        h->gumbel_pool = gp;
        const size_t T = (size_t)t->cap_trees;
        gp->cap_trees = t->cap_trees;
        gp->dev.npt = t->nodes_per_tree;
        CCX_CUDA(h, cudaMalloc(&gp->dev.vraw, T * t->nodes_per_tree * 8));
        CCX_CUDA(h, cudaMalloc(&gp->dev.g, T * GUMBEL_EDGES * 8));
        CCX_CUDA(h, cudaMalloc(&gp->dev.mp, T * 4));
        gp->bytes = T * ((size_t)t->nodes_per_tree * 8 + GUMBEL_EDGES * 8 + 4);
    }
    const int32_t m = h->gumbel_m;
    if (gp->table_m != m || gp->table_s != sims) {
        const int32_t rows = (m < GUMBEL_EDGES ? m : GUMBEL_EDGES) + 1, cols = sims > 0 ? sims : 1;
        int32_t *host = (int32_t *)calloc((size_t)rows * cols, 4);
        if (!host) return CCX_ERR_NOMEM;
        for (int32_t r = 0; r < rows; r++) ccx_considered_visits(r, sims, host + (size_t)r * cols);
        if (gp->table) { cudaFree(gp->table); gp->table = nullptr; }
        cudaError_t e = cudaMalloc(&gp->table, (size_t)rows * cols * 4);
        if (e == cudaSuccess) e = cudaMemcpy(gp->table, host, (size_t)rows * cols * 4, cudaMemcpyHostToDevice);
        free(host);
        if (e != cudaSuccess) return ccx_fail(h, e);
        gp->table_m = m; gp->table_s = sims;
        gp->dev.table = gp->table; gp->dev.rows = rows; gp->dev.cols = cols;
        gp->bytes = (size_t)gp->cap_trees * ((size_t)gp->dev.npt * 8 + GUMBEL_EDGES * 8 + 4) + (size_t)rows * cols * 4;
        h->epoch++;
    }
    gp->dev.m = m;
    gp->dev.scale = h->gumbel_scale; gp->dev.c_visit = h->gumbel_c_visit; gp->dev.c_scale = h->gumbel_c_scale;
    gp->dev.seed_lo = (u32)h->gumbel_seed; gp->dev.seed_hi = (u32)(h->gumbel_seed >> 32);
    return CCX_OK;
}

static inline const ccx_gumbel_dev &gumbel_dev(const ccx_handle *h) { return ((const ccx_gumbel_pool *)h->gumbel_pool)->dev; }

extern "C" {

int ccx_mcts_search(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t evaluator, int32_t num_itr, double cpuct,
                    double tau, int32_t pre_expand, const double *root_noise, int32_t noise_stride,
                    int32_t edges_per_tree, uint32_t *visits, double *pi, double *q, int32_t *n_nodes)
{
    if (!h || n < 0 || num_itr < 0 || !(tau > 0.0) || (n && (!roots || !visits))) return CCX_ERR_ARG;
    if (evaluator != EVAL_UNIFORM && evaluator != EVAL_HASH) return CCX_ERR_UNSUPPORTED;   // the net runs round-based
    if (h->gumbel) return CCX_ERR_UNSUPPORTED;
    if (root_noise && noise_stride < 1) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    int rc = trees_reserve(h, n, num_itr, edges_per_tree);
    if (rc) return rc;
    h->search_gen = h->pool_gen; h->search_n = n;
    unsigned grid = tree_blocks(n);
#define CCX_SEARCH(EV, TI) k_mcts_search<EV, TI><<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, (const u64 *)roots, n, num_itr, \
                                                                                                   cpuct, pre_expand, root_noise, noise_stride, h->jump_table)
    const bool ties = h->trees->tie_mode != 0;
    if (evaluator == EVAL_UNIFORM) { if (ties) CCX_SEARCH(EVAL_UNIFORM, true); else CCX_SEARCH(EVAL_UNIFORM, false); }
    else { if (ties) CCX_SEARCH(EVAL_HASH, true); else CCX_SEARCH(EVAL_HASH, false); }
#undef CCX_SEARCH
    CCX_LAUNCHED(h);
    k_mcts_finalize<<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, 1.0 / tau, visits, pi, q, n_nodes);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_set_tiebreak(ccx_handle *h, int32_t mode, uint64_t seed, int64_t uid0)
{
    if (!h || (mode != 0 && mode != 1)) return CCX_ERR_ARG;
    h->tie_mode = mode; h->tie_seed = seed; h->tie_uid0 = uid0;
    if (h->trees) {
        ccx_trees *t = h->trees;
        t->tie_mode = mode;                           // by-value kernel argument: selects the instantiation, keys the cached round graph
        const u32 tp[4] = {(u32)seed, (u32)(seed >> 32), (u32)(uint64_t)uid0, (u32)((uint64_t)uid0 >> 32)};
        CCX_CUDA(h, cudaMemcpyAsync(t->tie_params, tp, 16, cudaMemcpyHostToDevice, h->stream));     // in stream order with the searches
    }
    return CCX_OK;
}

int ccx_mcts_begin(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t num_itr, int32_t edges_per_tree, int32_t min_ply,
                   int32_t ply_parity)
{
    if (!h || n < 0 || num_itr < 0 || (n && !roots) || ply_parity < -1 || ply_parity > 1) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    int rc = trees_reserve(h, n, num_itr, edges_per_tree);
    if (rc) return rc;
    if (h->gumbel && (rc = gumbel_pool_reserve(h, num_itr > 0 ? num_itr - 1 : 0))) return rc;
    k_mcts_init<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, (const u64 *)roots, n, min_ply, ply_parity);
    CCX_LAUNCHED(h);
    h->search_gen = h->pool_gen; h->search_n = n;
    return CCX_OK;
}

int ccx_mcts_begin_reuse(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t num_itr, int32_t edges_per_tree, int32_t min_ply,
                         int32_t ply_parity, int32_t carry, const int64_t *prev, const double *root_noise, int32_t noise_stride,
                         int32_t noise_normalize, int32_t *reused)
{
    if (!h || n < 0 || num_itr < 0 || (n && !roots) || ply_parity < -1 || ply_parity > 1 || carry < 0) return CCX_ERR_ARG;
    if (root_noise && noise_stride < 1) return CCX_ERR_ARG;
    if (h->gumbel) return CCX_ERR_UNSUPPORTED;
    const int64_t E = edges_per_tree > 0 ? edges_per_tree : 64 * ((int64_t)num_itr + 1);
    if ((1 + (int64_t)carry) * (E > num_itr + 2 ? E : num_itr + 2) > 0x7FFFFFFF) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    int rc = trees_reserve(h, n, num_itr, edges_per_tree, carry);
    if (rc) return rc;
    const int64_t n_prev = h->search_gen == h->pool_gen ? h->search_n : 0;     // trees of another generation are no source
    const int32_t lim_nodes = carry * (num_itr + 2), lim_edges = (int32_t)(carry * E);
    if ((rc = reuse_pool_reserve(h, lim_nodes > 0 ? lim_nodes : 1, lim_edges > 0 ? lim_edges : 1))) return rc;
    const ccx_reuse_pool &rp = *(const ccx_reuse_pool *)h->reuse_pool;
    const unsigned grid = tree_blocks(n), threads = 32 * MCTS_WARPS_PER_BLOCK;
    k_mcts_reuse_match<<<grid, threads, 0, h->stream>>>(*h->trees, (const u64 *)roots, n, n_prev, prev, min_ply, ply_parity,
                                                        (int64_t)carry * (num_itr + 1), rp.rec);
    CCX_LAUNCHED(h);
    k_mcts_reuse_gather<<<grid, threads, 0, h->stream>>>(*h->trees, rp.scratch, rp.qsrc, n, rp.rec, lim_nodes, lim_edges, root_noise,
                                                         noise_stride, noise_normalize);
    CCX_LAUNCHED(h);
    k_mcts_reuse_commit<<<(unsigned)n, REUSE_COMMIT_THREADS, 0, h->stream>>>(*h->trees, rp.scratch, (const u64 *)roots, n, rp.rec, min_ply, ply_parity,
                                                         reused);
    CCX_LAUNCHED(h);
    h->search_gen = h->pool_gen; h->search_n = n;
    return CCX_OK;
}

int ccx_mcts_select(ccx_handle *h, int64_t n, double cpuct, uint64_t *leaf_state)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || (n && !leaf_state)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    if (h->gumbel) {
        if (!h->gumbel_pool) return CCX_ERR_STATE;                   // no begin in the mode on these trees
        k_mcts_select_gumbel<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, gumbel_dev(h), n, (u64 *)leaf_state);
        CCX_LAUNCHED(h);
        return CCX_OK;
    }
    if (h->trees->tie_mode) k_mcts_select<true><<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, cpuct, (u64 *)leaf_state);
    else k_mcts_select<false><<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, cpuct, (u64 *)leaf_state);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_expand_backup(ccx_handle *h, int64_t n, const double *p, const double *v, const double *root_noise,
                           int32_t noise_stride, int32_t noise_normalize)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || (n && (!p || !v))) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    if (h->gumbel) {
        if (root_noise) return CCX_ERR_UNSUPPORTED;
        if (!h->gumbel_pool) return CCX_ERR_STATE;
        k_mcts_expand_backup_gumbel<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, gumbel_dev(h), n, p, v,
                                                                                               h->jump_table);
        CCX_LAUNCHED(h);
        return CCX_OK;
    }
    k_mcts_expand_backup<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, p, v, root_noise, noise_stride, noise_normalize, h->jump_table);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

}  // extern "C"

// round r of trees [t0, t0 + nq) with a mirror-symmetric net evaluation (ccx_net_set_symmetry), as the launches of
// run_net_rounds below
template <int SYM>
static void launch_round_sym(ccx_handle *h, cudaStream_t st, int r, int32_t rounds, int64_t t0, int64_t nq, double cpuct,
                             const double *nz, int32_t noise_stride, int32_t noise_normalize, uint8_t *planes, const float *logits,
                             const float *value)
{
    const unsigned grid = tree_blocks(nq), threads = 32 * MCTS_WARPS_PER_BLOCK;
    const u32 k0 = (u32)h->sym_seed, k1 = (u32)(h->sym_seed >> 32);
    const bool ties = h->trees->tie_mode != 0;
    if (h->gumbel) {
        const ccx_gumbel_dev &gd = gumbel_dev(h);
        if (r == 0) k_mcts_select_encode_gumbel_sym<SYM><<<grid, threads, 0, st>>>(*h->trees, gd, t0, nq, planes, k0, k1);
        else if (r < rounds) k_mcts_round_gumbel_sym<SYM><<<grid, threads, 0, st>>>(*h->trees, gd, t0, nq, logits, value, planes,
                                                                                  h->jump_table, k0, k1);
        else k_mcts_softmax_expand_backup_gumbel_sym<SYM><<<grid, threads, 0, st>>>(*h->trees, gd, t0, nq, logits, value, h->jump_table,
                                                                                  k0, k1);
    } else if (r == 0) {
        if (ties) k_mcts_select_encode_sym<true, SYM><<<grid, threads, 0, st>>>(*h->trees, t0, nq, cpuct, planes, k0, k1);
        else k_mcts_select_encode_sym<false, SYM><<<grid, threads, 0, st>>>(*h->trees, t0, nq, cpuct, planes, k0, k1);
    } else if (r < rounds) {
        const double *noise = r == 1 ? nz : nullptr;
        if (ties) k_mcts_round_sym<true, SYM><<<grid, threads, 0, st>>>(*h->trees, t0, nq, cpuct, logits, value, noise, noise_stride,
                                                                       noise_normalize, planes, h->jump_table, k0, k1);
        else k_mcts_round_sym<false, SYM><<<grid, threads, 0, st>>>(*h->trees, t0, nq, cpuct, logits, value, noise, noise_stride,
                                                                   noise_normalize, planes, h->jump_table, k0, k1);
    } else {
        k_mcts_softmax_expand_backup_sym<SYM><<<grid, threads, 0, st>>>(*h->trees, t0, nq, logits, value, rounds == 1 ? nz : nullptr,
                                                                       noise_stride, noise_normalize, h->jump_table, k0, k1);
    }
}

// a leaf-parallel round (as the launches of run_net_leaves_rounds below) with a mirror-symmetric net evaluation
template <int SYM>
static void launch_leaves_sym(ccx_handle *h, cudaStream_t st, int r, const ccx_leaf_pool &lp, int64_t t0, int64_t nq, int32_t leaves,
                              double cpuct, int32_t sims, int budget, const double *root_noise, int32_t noise_stride, int32_t noise_normalize,
                              uint8_t *planes, const float *logits, const float *value)
{
    const unsigned grid = (unsigned)nq, threads = 32 * leaves;
    const size_t smem_select = (size_t)leaves * 352, smem_round = (size_t)leaves * (296 * 8 + 352);
    const u32 k0 = (u32)h->sym_seed, k1 = (u32)(h->sym_seed >> 32);
    const bool ties = h->trees->tie_mode != 0;
    if (r == 0) {
        if (ties) k_mcts_select_leaves_sym<true, SYM><<<grid, threads, smem_select, st>>>(*h->trees, lp, t0, leaves, cpuct, sims, planes, k0, k1);
        else k_mcts_select_leaves_sym<false, SYM><<<grid, threads, smem_select, st>>>(*h->trees, lp, t0, leaves, cpuct, sims, planes, k0, k1);
    } else {
        if (ties) k_mcts_round_leaves_sym<true, SYM><<<grid, threads, smem_round, st>>>(*h->trees, lp, t0, leaves, cpuct, logits, value, root_noise,
                                                                                       noise_stride, noise_normalize, planes, h->jump_table,
                                                                                       budget, k0, k1);
        else k_mcts_round_leaves_sym<false, SYM><<<grid, threads, smem_round, st>>>(*h->trees, lp, t0, leaves, cpuct, logits, value, root_noise,
                                                                                   noise_stride, noise_normalize, planes, h->jump_table,
                                                                                   budget, k0, k1);
    }
}

extern "C" {

// the round loop itself, issued on h->stream (and h->stream2 for the second half of a split batch).  The net batch holds
// R = SymRows rows per tree (two in the mean-of-both-orientations mode); the split threshold counts rows.
static int run_net_rounds(ccx_handle *h, int64_t n, int32_t rounds, double cpuct, const double *root_noise, int32_t noise_stride,
                          int32_t noise_normalize)
{
    uint8_t *planes; float *logits, *value;
    int rc;
    const int64_t R = h->sym_mode == SYM_MEAN ? 2 : 1, rows = n * R;
    if ((rc = ccx_net_scratch(h, rows, &planes, &logits, &value))) return rc;
    // Two halves of the batch run as two independent round pipelines on two streams: trees are independent, and the
    // low-occupancy stretches of one half (the tail of its tree kernel = the deepest trees, the last tile of its trunk kernel)
    // are filled by the other half's kernels.  Same trees as the single-stream order, bit for bit.
    static const bool no_split = getenv("CCX_NO_SPLIT") != nullptr;
    // batch size from which the two-half pipeline is used: 8,192 in the 16-bit mode; 16,384 in the accurate mode, whose three-context
    // trunk loses more on a halved batch (r02h, accurate mode: 8,192 slots 52.2 ms unsplit / 53.7 split, 16,384 slots 100.8 / 98.3)
    static const int64_t split_env = getenv("CCX_SPLIT_MIN") ? atoll(getenv("CCX_SPLIT_MIN")) : -1;
    const int64_t split_min = split_env >= 0 ? split_env : h->net_mode == 2 ? 16384 : 8192;
    const bool split = !no_split && (h->net_mode == 1 || h->net_mode == 2) && rows >= split_min;     // measured (16-bit mode): 16,384 slots 65.1 -> 62.2 ms per ply; no gain at 4,096
    int64_t part_n[2] = {split ? (n / 2) & ~(int64_t)127 : n, 0};          // halves start on a 128-position tile of the net's scratch
    part_n[1] = n - part_n[0];
    cudaStream_t streams[2] = {h->stream, h->stream};
    if (split) {
        if (!h->stream2) {
            CCX_CUDA(h, cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
            CCX_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
            CCX_CUDA(h, cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
        }
        streams[1] = h->stream2;
        CCX_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
        CCX_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
    }
    // make sure the evaluator's internal scratch covers the whole batch before two streams share it
    if (h->net_mode == 1 && (rc = ccx_net_forward_tc_on(h, h->stream, rows, 0, 0, planes, logits, value))) return rc;
    if (h->net_mode == 2 && (rc = ccx_net_forward_acc_on(h, h->stream, rows, 0, 0, planes, logits, value, ccx_net_pold_bias(h)))) return rc;
    const int parts = split ? 2 : 1;
    // round r: [r == 0: select+encode | r > 0: finish round r-1's leaf, then select+encode] -> net; one last finish at the end.
    // Tried and dropped (r01c): programmatic dependent launch for the three kernels of a round (prologues before
    // griddepcontrol.wait, launch_dependents at kernel start) — 23.8 ms per 4,096-slot ply against 21.3 ms without, and
    // 94 ms against 73 ms at 16,384 slots: early-scheduled dependent CTAs take SM slots from the producer's later waves.
    for (int r = 0; r <= rounds; r++) {
        for (int q = 0; q < parts; q++) {
            const int64_t t0 = q ? part_n[0] : 0, nq = part_n[q];
            if (nq == 0) continue;
            cudaStream_t st = streams[q];
            const unsigned grid = tree_blocks(nq);
            const double *nz = root_noise;
            const bool ties = h->trees->tie_mode != 0;
            if (h->sym_mode == SYM_RANDOM) {
                launch_round_sym<SYM_RANDOM>(h, st, r, rounds, t0, nq, cpuct, nz, noise_stride, noise_normalize, planes, logits, value);
            } else if (h->sym_mode == SYM_MEAN) {
                launch_round_sym<SYM_MEAN>(h, st, r, rounds, t0, nq, cpuct, nz, noise_stride, noise_normalize, planes, logits, value);
            } else if (h->gumbel) {
                const ccx_gumbel_dev &gd = gumbel_dev(h);
                if (r == 0) k_mcts_select_encode_gumbel<<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, gd, t0, nq, planes);
                else if (r < rounds) k_mcts_round_gumbel<<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, gd, t0, nq, logits, value,
                                                                                                   planes, h->jump_table);
                else k_mcts_softmax_expand_backup_gumbel<<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, gd, t0, nq, logits, value,
                                                                                                   h->jump_table);
            } else if (r == 0) {
                if (ties) k_mcts_select_encode<true><<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, t0, nq, cpuct, planes);
                else k_mcts_select_encode<false><<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, t0, nq, cpuct, planes);
            } else if (r < rounds) {
                if (ties) k_mcts_round<true><<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, t0, nq, cpuct, logits, value, r == 1 ? nz : nullptr,
                                                                                       noise_stride, noise_normalize, planes, h->jump_table);
                else k_mcts_round<false><<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, t0, nq, cpuct, logits, value, r == 1 ? nz : nullptr,
                                                                                     noise_stride, noise_normalize, planes, h->jump_table);
            }
            else
                k_mcts_softmax_expand_backup<<<grid, 32 * MCTS_WARPS_PER_BLOCK, 0, st>>>(*h->trees, t0, nq, logits, value,
                                                                                         rounds == 1 ? nz : nullptr, noise_stride,
                                                                                         noise_normalize, h->jump_table);
            CCX_LAUNCHED(h);
            if (r < rounds) {
                const int64_t p0 = t0 * R, pn = nq * R;
                if (h->net_mode == 1) rc = ccx_net_forward_tc_on(h, st, rows, p0, pn, planes + p0 * 343, logits + p0 * 294, value + p0);
                else if (h->net_mode == 2) rc = ccx_net_forward_acc_on(h, st, rows, p0, pn, planes + p0 * 343, logits + p0 * 294, value + p0, ccx_net_pold_bias(h));
                else rc = ccx_net_forward_active(h, pn, planes + p0 * 343, logits + p0 * 294, value + p0);
                if (rc) return rc;
            }
        }
    }
    if (split) {
        CCX_CUDA(h, cudaEventRecord(h->ev_join, h->stream2));
        CCX_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));
    }
    return CCX_OK;
}

// the leaf-parallel round loop: as run_net_rounds with a net batch of n * leaves positions (slot i*leaves + k; R = SymRows
// rows per slot); the two-half split is decided on rows and cuts between trees
static int run_net_leaves_rounds(ccx_handle *h, int64_t n, int32_t sims, int32_t leaves, double cpuct, const double *root_noise,
                                 int32_t noise_stride, int32_t noise_normalize)
{
    const int64_t R = h->sym_mode == SYM_MEAN ? 2 : 1;
    const int64_t np = n * leaves * R;
    const int32_t rounds = 1 + (sims - 1 + leaves - 1) / leaves;        // first round: one selection per unexpanded root
    uint8_t *planes; float *logits, *value;
    int rc;
    if ((rc = ccx_net_scratch(h, np, &planes, &logits, &value))) return rc;
    static const bool no_split = getenv("CCX_NO_SPLIT") != nullptr;
    static const int64_t split_env = getenv("CCX_SPLIT_MIN") ? atoll(getenv("CCX_SPLIT_MIN")) : -1;
    const int64_t split_min = split_env >= 0 ? split_env : h->net_mode == 2 ? 16384 : 8192;
    const int64_t half = (n / 2) & ~(int64_t)127;                      // 128 trees: the halves start on a 128-position tile
    const bool split = !no_split && (h->net_mode == 1 || h->net_mode == 2) && np >= split_min && half > 0;
    int64_t part_n[2] = {split ? half : n, 0};
    part_n[1] = n - part_n[0];
    cudaStream_t streams[2] = {h->stream, h->stream};
    if (split) {
        if (!h->stream2) {
            CCX_CUDA(h, cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
            CCX_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
            CCX_CUDA(h, cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
        }
        streams[1] = h->stream2;
        CCX_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
        CCX_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
    }
    if (h->net_mode == 1 && (rc = ccx_net_forward_tc_on(h, h->stream, np, 0, 0, planes, logits, value))) return rc;
    if (h->net_mode == 2 && (rc = ccx_net_forward_acc_on(h, h->stream, np, 0, 0, planes, logits, value, ccx_net_pold_bias(h)))) return rc;
    const ccx_leaf_pool lp = *(const ccx_leaf_pool *)h->leaf_pool;
    const bool ties = h->trees->tie_mode != 0;
    const unsigned threads = 32 * leaves;
    const size_t smem_select = (size_t)leaves * 352, smem_round = (size_t)leaves * (296 * 8 + 352);
    for (int r = 0; r <= rounds; r++) {
        for (int q = 0; q < (split ? 2 : 1); q++) {
            const int64_t t0 = q ? part_n[0] : 0, nq = part_n[q];
            if (nq == 0) continue;
            cudaStream_t st = streams[q];
            const unsigned grid = (unsigned)nq;
            const int budget = r < rounds ? -1 : 0;
            if (h->sym_mode == SYM_RANDOM) {
                launch_leaves_sym<SYM_RANDOM>(h, st, r, lp, t0, nq, leaves, cpuct, sims, budget, root_noise, noise_stride, noise_normalize,
                                              planes, logits, value);
            } else if (h->sym_mode == SYM_MEAN) {
                launch_leaves_sym<SYM_MEAN>(h, st, r, lp, t0, nq, leaves, cpuct, sims, budget, root_noise, noise_stride, noise_normalize,
                                            planes, logits, value);
            } else if (r == 0) {
                if (ties) k_mcts_select_leaves<true, true><<<grid, threads, smem_select, st>>>(*h->trees, lp, t0, leaves, cpuct, sims, planes,
                                                                                             nullptr, 0);
                else k_mcts_select_leaves<false, true><<<grid, threads, smem_select, st>>>(*h->trees, lp, t0, leaves, cpuct, sims, planes,
                                                                                           nullptr, 0);
            } else {
                if (ties) k_mcts_round_leaves<true><<<grid, threads, smem_round, st>>>(*h->trees, lp, t0, leaves, cpuct, logits, value, root_noise,
                                                                             noise_stride, noise_normalize, planes, h->jump_table, budget);
                else k_mcts_round_leaves<false><<<grid, threads, smem_round, st>>>(*h->trees, lp, t0, leaves, cpuct, logits, value, root_noise,
                                                                         noise_stride, noise_normalize, planes, h->jump_table, budget);
            }
            CCX_LAUNCHED(h);
            if (r < rounds) {
                const int64_t p0 = t0 * leaves * R, pn = nq * leaves * R;
                if (h->net_mode == 1) rc = ccx_net_forward_tc_on(h, st, np, p0, pn, planes + p0 * 343, logits + p0 * 294, value + p0);
                else if (h->net_mode == 2) rc = ccx_net_forward_acc_on(h, st, np, p0, pn, planes + p0 * 343, logits + p0 * 294, value + p0,
                                                                       ccx_net_pold_bias(h));
                else rc = ccx_net_forward_active(h, pn, planes + p0 * 343, logits + p0 * 294, value + p0);
                if (rc) return rc;
            }
        }
    }
    if (split) {
        CCX_CUDA(h, cudaEventRecord(h->ev_join, h->stream2));
        CCX_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));
    }
    return CCX_OK;
}

// One search = rounds x (tree kernel, trunk, policy dense): ~530 dependent launches for 175 simulations.  The loop is the same
// from ply to ply (same buffers, same arguments), so it is captured once into a CUDA graph and replayed: 19.45 -> 18.25 ms per
// 4,096-tree search in the 16-bit mode and 33.4 -> 32.2 ms in the accurate mode on B200 (the gaps between dependent kernels
// shrink).  Life cycle per argument set: first call runs directly (and performs every lazy allocation), second call is
// captured on an internal stream and instantiated, later calls replay.  `epoch` + the by-value tree descriptor + the call's
// arguments are the cache key; CCX_NO_GRAPH=1 switches the replay off.
// The leaf-parallel loop is cached the same way; its key adds `leaves` and the per-leaf buffers, and `rounds` holds its
// selection count.
static bool round_graph_matches(const ccx_round_graph *g, const ccx_handle *h, int64_t n, int32_t rounds, int32_t leaves, double cpuct,
                                const double *noise, int32_t stride, int32_t normalize)
{
    return g->seen && g->epoch == h->epoch && g->n == n && g->rounds == rounds && g->leaves == leaves && g->cpuct == cpuct &&
           g->noise == noise && g->stride == stride && g->normalize == normalize && memcmp(&g->trees, h->trees, sizeof(ccx_trees)) == 0 &&
           (leaves == 1 || memcmp(&g->pool, h->leaf_pool, sizeof(ccx_leaf_pool)) == 0) && g->gumbel == h->gumbel &&
           (!h->gumbel || memcmp(&g->gdev, &gumbel_dev(h), sizeof(ccx_gumbel_dev)) == 0);
}

static int run_any_rounds(ccx_handle *h, int64_t n, int32_t rounds, int32_t leaves, double cpuct, const double *root_noise,
                          int32_t noise_stride, int32_t noise_normalize)
{
    return leaves == 1 ? run_net_rounds(h, n, rounds, cpuct, root_noise, noise_stride, noise_normalize)
                       : run_net_leaves_rounds(h, n, rounds, leaves, cpuct, root_noise, noise_stride, noise_normalize);
}

// leaves == 1: `rounds` one-leaf rounds; leaves > 1: `rounds` selections in leaf-parallel rounds
static int run_net_cached(ccx_handle *h, int64_t n, int32_t rounds, int32_t leaves, double cpuct, const double *root_noise,
                          int32_t noise_stride, int32_t noise_normalize)
{
    static const bool no_graph = getenv("CCX_NO_GRAPH") != nullptr;
    cudaStreamCaptureStatus user_capture = cudaStreamCaptureStatusNone;
    const int32_t launched_rounds = leaves == 1 ? rounds : 1 + (rounds - 1 + leaves - 1) / leaves;
    if (no_graph || h->graph_off || launched_rounds < 8 || cudaStreamIsCapturing(h->stream, &user_capture) != cudaSuccess ||
        user_capture != cudaStreamCaptureStatusNone) {
        cudaGetLastError();
        return run_any_rounds(h, n, rounds, leaves, cpuct, root_noise, noise_stride, noise_normalize);
    }
    ccx_round_graph *g = (ccx_round_graph *)h->round_graph;
    if (!g) {
        g = new (std::nothrow) ccx_round_graph();
        if (!g) return CCX_ERR_NOMEM;
        h->round_graph = g;
    }
    if (!round_graph_matches(g, h, n, rounds, leaves, cpuct, root_noise, noise_stride, noise_normalize)) {
        // new argument set: run directly once (lazy allocations happen here), remember the key as it stands afterwards
        if (g->exec) { cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
        g->seen = false;
        int rc = run_any_rounds(h, n, rounds, leaves, cpuct, root_noise, noise_stride, noise_normalize);
        if (rc) return rc;
        g->seen = true; g->epoch = h->epoch; g->n = n; g->rounds = rounds; g->leaves = leaves; g->cpuct = cpuct; g->noise = root_noise;
        g->stride = noise_stride; g->normalize = noise_normalize;
        memcpy(&g->trees, h->trees, sizeof(ccx_trees));
        if (leaves > 1) memcpy(&g->pool, h->leaf_pool, sizeof(ccx_leaf_pool));
        g->gumbel = h->gumbel;
        if (h->gumbel) memcpy(&g->gdev, &gumbel_dev(h), sizeof(ccx_gumbel_dev));
        return CCX_OK;
    }
    if (!g->exec) {
        if (!h->cap_stream) CCX_CUDA(h, cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
        cudaStream_t user = h->stream;
        const int64_t before = h->launches;
        cudaGraph_t graph = nullptr;
        static const bool debug = getenv("CCX_GRAPH_DEBUG") != nullptr;
        cudaError_t ce = cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal);
        bool ok = ce == cudaSuccess;
        if (!ok && debug) fprintf(stderr, "ccx graph: begin capture: %s\n", cudaGetErrorString(ce));
        if (ok) {
            h->stream = h->cap_stream;
            int rc = run_any_rounds(h, n, rounds, leaves, cpuct, root_noise, noise_stride, noise_normalize);
            h->stream = user;
            ce = cudaStreamEndCapture(h->cap_stream, &graph);
            ok = ce == cudaSuccess && rc == CCX_OK && graph != nullptr;
            if (!ok && debug) fprintf(stderr, "ccx graph: capture rc %d, end capture: %s (%s)\n", rc, cudaGetErrorString(ce), h->cuda_err);
        }
        if (ok) {
            ce = cudaGraphInstantiate(&g->exec, graph, 0);
            ok = ce == cudaSuccess;
            if (!ok && debug) fprintf(stderr, "ccx graph: instantiate: %s\n", cudaGetErrorString(ce));
        }
        if (graph) cudaGraphDestroy(graph);
        g->launches = h->launches - before;
        h->launches = before;
        if (debug && ok && g->epoch != h->epoch) fprintf(stderr, "ccx graph: epoch moved during capture\n");
        if (!ok || g->epoch != h->epoch) {                 // capture refused or something was reallocated under it: no graphs on this handle
            cudaGetLastError();
            if (g->exec) { cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
            g->seen = false;
            h->graph_off = 1;
            return run_any_rounds(h, n, rounds, leaves, cpuct, root_noise, noise_stride, noise_normalize);
        }
    }
    CCX_CUDA(h, cudaGraphLaunch(g->exec, h->stream));
    h->launches += g->launches;
    h->graph_replays++;
    return CCX_OK;
}

int ccx_mcts_run_net(ccx_handle *h, int64_t n, int32_t rounds, double cpuct, const double *root_noise, int32_t noise_stride,
                     int32_t noise_normalize)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || rounds < 0) return CCX_ERR_ARG;
    if (root_noise && noise_stride < 1) return CCX_ERR_ARG;
    if (n == 0 || rounds == 0) return CCX_OK;
    if (h->gumbel && root_noise) return CCX_ERR_UNSUPPORTED;
    if (h->gumbel && !h->gumbel_pool) return CCX_ERR_STATE;
    return run_net_cached(h, n, rounds, 1, cpuct, root_noise, noise_stride, noise_normalize);
}

int ccx_mcts_run_net_leaves(ccx_handle *h, int64_t n, int32_t sims, int32_t leaves, double cpuct, const double *root_noise,
                            int32_t noise_stride, int32_t noise_normalize)
{
    if (leaves < 1 || leaves > CCX_MAX_LEAVES) return CCX_ERR_ARG;
    if (leaves == 1) return ccx_mcts_run_net(h, n, sims, cpuct, root_noise, noise_stride, noise_normalize);
    if (h && h->gumbel) return CCX_ERR_UNSUPPORTED;
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || sims < 0) return CCX_ERR_ARG;
    if (root_noise && noise_stride < 1) return CCX_ERR_ARG;
    if (n == 0 || sims == 0) return CCX_OK;
    int rc = leaf_pool_reserve(h, leaves);
    if (rc) return rc;
    return run_net_cached(h, n, sims, leaves, cpuct, root_noise, noise_stride, noise_normalize);
}

int ccx_mcts_leaf_budget(ccx_handle *h, int64_t n, int32_t leaves, int32_t sims)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || leaves < 1 || leaves > CCX_MAX_LEAVES || sims < 0) return CCX_ERR_ARG;
    if (leaves == 1 || n == 0) return CCX_OK;            // one-leaf rounds make one selection per call
    int rc = leaf_pool_reserve(h, leaves);
    if (rc) return rc;
    k_mcts_leaf_budget<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(*(const ccx_leaf_pool *)h->leaf_pool, n, sims);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_select_leaves(ccx_handle *h, int64_t n, int32_t leaves, double cpuct, uint64_t *leaf_state)
{
    if (leaves < 1 || leaves > CCX_MAX_LEAVES) return CCX_ERR_ARG;
    if (leaves == 1) return ccx_mcts_select(h, n, cpuct, leaf_state);
    if (h && h->gumbel) return CCX_ERR_UNSUPPORTED;
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || (n && !leaf_state)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    int rc = leaf_pool_reserve(h, leaves);
    if (rc) return rc;
    const ccx_leaf_pool &lp = *(const ccx_leaf_pool *)h->leaf_pool;
    if (h->trees->tie_mode)
        k_mcts_select_leaves<true, false><<<(unsigned)n, 32 * leaves, 0, h->stream>>>(*h->trees, lp, 0, leaves, cpuct, -1, nullptr,
                                                                                    (u64 *)leaf_state, n * leaves);
    else
        k_mcts_select_leaves<false, false><<<(unsigned)n, 32 * leaves, 0, h->stream>>>(*h->trees, lp, 0, leaves, cpuct, -1, nullptr,
                                                                                     (u64 *)leaf_state, n * leaves);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_expand_backup_leaves(ccx_handle *h, int64_t n, int32_t leaves, const double *p, const double *v, const double *root_noise,
                                  int32_t noise_stride, int32_t noise_normalize)
{
    if (leaves < 1 || leaves > CCX_MAX_LEAVES) return CCX_ERR_ARG;
    if (leaves == 1) return ccx_mcts_expand_backup(h, n, p, v, root_noise, noise_stride, noise_normalize);
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || (n && (!p || !v))) return CCX_ERR_ARG;
    if (root_noise && noise_stride < 1) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    ccx_leaf_pool *lp = (ccx_leaf_pool *)h->leaf_pool;
    if (!lp || lp->cap_leaves < leaves) return CCX_ERR_ARG;      // no ccx_mcts_select_leaves round on these trees
    k_mcts_backup_leaves<<<(unsigned)n, 32 * leaves, 0, h->stream>>>(*h->trees, *lp, 0, leaves, p, v, root_noise, noise_stride,
                                                                            noise_normalize, h->jump_table);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_finalize(ccx_handle *h, int64_t n, double tau, uint32_t *visits, double *pi, double *q, int32_t *n_nodes)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || !(tau > 0.0) || (n && !visits)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_mcts_finalize<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, 1.0 / tau, visits, pi, q, n_nodes);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_get_root(ccx_handle *h, int64_t n, int32_t stride, int32_t *n_edges, uint16_t *moves, uint32_t *N, double *W,
                      double *P)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || stride < 1 || (n && (!n_edges || !moves || !N || !W || !P)))
        return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_mcts_get_root<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, stride, n_edges, moves, N, W, P);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_mcts_set_root_priors(ccx_handle *h, int64_t n, int32_t stride, const double *P)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || stride < 1 || (n && !P)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_mcts_set_root_priors<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, n, stride, P);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int64_t ccx_mcts_pool_bytes(const ccx_handle *h)
{
    if (!h || !h->trees) return 0;
    const ccx_leaf_pool *lp = (const ccx_leaf_pool *)h->leaf_pool;
    const ccx_reuse_pool *rp = (const ccx_reuse_pool *)h->reuse_pool;
    const ccx_gumbel_pool *gp = (const ccx_gumbel_pool *)h->gumbel_pool;
    return (int64_t)(h->trees->bytes + (lp ? lp->bytes : 0) + (rp ? rp->bytes : 0) + (gp ? gp->bytes : 0));
}

int ccx_mcts_set_gumbel(ccx_handle *h, int32_t enabled, int32_t considered, double scale, double c_visit, double c_scale,
                        uint64_t seed)
{
    if (!h) return CCX_ERR_ARG;
    if (enabled && (considered < 1 || !(scale >= 0.0) || !(c_visit >= 0.0) || !(c_scale >= 0.0) || scale > 1e300 ||
                    c_visit > 1e300 || c_scale > 1e300))
        return CCX_ERR_ARG;
    h->gumbel = enabled != 0;
    if (enabled) {
        h->gumbel_m = considered; h->gumbel_scale = scale; h->gumbel_c_visit = c_visit; h->gumbel_c_scale = c_scale;
        h->gumbel_seed = seed;
    }
    return CCX_OK;
}

int ccx_mcts_finalize_gumbel(ccx_handle *h, int64_t n, uint32_t *visits, double *pi, double *q, int32_t *action, int32_t *n_nodes)
{
    if (!h || !h->trees || n < 0 || n > h->trees->cap_trees || (n && !visits)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    if (!h->gumbel_pool) return CCX_ERR_STATE;
    k_mcts_finalize_gumbel<<<tree_blocks(n), 32 * MCTS_WARPS_PER_BLOCK, 0, h->stream>>>(*h->trees, gumbel_dev(h), n, visits, pi, q,
                                                                                      action, n_nodes);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

}  // extern "C"
