/*
 * ccx.h — C-ABI of the B200-native batched Chinese Checkers engine (libccx.so).
 *
 * The reference (kenziyuliu/ChineseCheckersAgent) is pure Python and has no FFI layer; its boundary is
 * the Python object surface (SURVEY.md §8b).  Each entry point below replaces one reference function
 * for a BATCH of independent games and cites the reference file:line it stands in for.  The Python
 * mirror of the reference interface (chinesecheckersagent_b200/{board,utils,MCTS,player,game,selfplay}.py)
 * is a thin ctypes layer over these symbols; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the function name contains `_host`
 *   - every call is enqueued on the handle's stream (ccx_set_stream) and is asynchronous with
 *     respect to the host, except the `_host` variants, which return after their results are in the
 *     caller's host buffers
 *   - return value: 0 = CCX_OK, negative = error (ccx_strerror); never throws, never aborts
 *   - no global mutable state; one handle per (device, stream) user; handles are thread-compatible
 *
 * State layout ("SoA words"): uint64 state[CCX_STATE_WORDS][n], plane-major (word k of game i at
 * state[k*n + i]) so that consecutive threads read consecutive 8-byte words (coalesced).
 *   cell index  = 8*row + col   (row, col in 0..6 — the reference's numpy indices, board.py:20-26);
 *                 row stride 8 leaves guard bits so that direction shifts never wrap.
 *   word 0  OCC1   bitboard of player 1's checkers            (board.py:19-26 plane 0 == 1)
 *   word 1  OCC2   bitboard of player 2's checkers            (plane 0 == 2)
 *   word 2  CELLS1 byte id (0..5) = cell of player 1's checker `id`   (board.py:42-44 checkers_pos[1])
 *   word 3  CELLS2 same for player 2                                   (board.py:45-46)
 *   word 4  META   byte0 last move from, byte1 last move to, byte2/3 the move before (0xFF = none)
 *                  (board.py:246-248 hist_moves[-1], [-2]); bytes 4-5 plies played (uint16);
 *                  byte 6 side to move (0 = PLAYER_ONE, 1 = PLAYER_TWO); byte 7 status (CCX_ST_*)
 *   word 5  HIST_LO destinations of the last 8 plies, byte 0 most recent, 0xFF = none
 *   word 6  HIST_HI destinations of plies 9..16 ago      (board.py:54 hist_moves / game.py:60,73-75)
 *   word 7  AUX    self-play bookkeeping (selfplay.py:19-23): bytes 0-1 num_useless_moves,
 *                  byte 2/3 player_progresses[0/1], bytes 4-5 recorded plies
 * The env step reads and writes words 0-4 (40 B each way = the 80 B/step algorithmic traffic).
 */
#ifndef CCX_H
#define CCX_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCX_ABI_VERSION 2
#define CCX_STATE_WORDS 8
#define CCX_NUM_CHECKERS 6          /* config.py:8  */
#define CCX_BOARD_W 7               /* config.py:10 */
#define CCX_NUM_ACTIONS 294         /* utils.py:164-171: id*49 + r*7 + c */
#define CCX_TRACE_WORDS 12

enum { CCX_OK = 0, CCX_ERR_ARG = -1, CCX_ERR_CUDA = -2, CCX_ERR_NOMEM = -3, CCX_ERR_STATE = -4,
       CCX_ERR_UNSUPPORTED = -5, CCX_ERR_OVERFLOW = -6 };
/* status byte of META */
enum { CCX_ST_RUNNING = 0, CCX_ST_WON_P1 = 1, CCX_ST_WON_P2 = 2, CCX_ST_REPETITION = 3,
       CCX_ST_MOVE_LIMIT = 4, CCX_ST_NO_MOVES = 5,
       CCX_ST_OVERFLOW = 6 /* engine-side stop, no reference counterpart: the search's edge pool or the record ring overflowed */,
       /* opt-in self-play resignation (ccx_selfplay_resign), no reference counterpart: the side to move resigned, the other won */
       CCX_ST_RESIGN_WON_P1 = 7, CCX_ST_RESIGN_WON_P2 = 8 };
enum { CCX_RESET_START = 0, CCX_RESET_RANDOMISED = 1 };
enum { CCX_DTYPE_U8 = 0, CCX_DTYPE_BF16 = 1, CCX_DTYPE_F32 = 2 };

typedef struct ccx_handle ccx_handle;

int         ccx_abi_version(void);
const char *ccx_strerror(int code);
/* last CUDA error string seen by this handle (empty if none) */
const char *ccx_last_cuda_error(const ccx_handle *h);

int ccx_create(int device_ordinal, ccx_handle **out);
int ccx_destroy(ccx_handle *h);
/* cuda_stream is a cudaStream_t passed as void*; NULL = the legacy default stream */
int ccx_set_stream(ccx_handle *h, void *cuda_stream);
int ccx_synchronize(ccx_handle *h);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches) */
int64_t ccx_launch_count(const ccx_handle *h);
/* searches served by replaying the cached CUDA graph of the round loop (ccx_mcts_run_net); diagnostics */
int64_t ccx_graph_replays(const ccx_handle *h);

/* Board() / Board(randomised=True)  — board.py:10-57, 61-85.  RANDOMISED draws 12 distinct cells with
 * Philox4x32-10 keyed by (seed, game_id0 + i); the first six go to player 1 ids 0..5. */
int ccx_reset(ccx_handle *h, int64_t n, uint64_t *state, int mode, uint64_t seed, int64_t game_id0);

/* Board.get_valid_moves(side to move) — board.py:139-222.  dest_masks[id*n + i] = bitboard of the
 * legal destinations of checker `id` (canonical order = ascending bit = ascending r*7+c). */
int ccx_movegen(ccx_handle *h, int64_t n, const uint64_t *state, uint64_t *dest_masks);

/* Board.place(side to move, from, to) -> check_win() — board.py:226-250, 89-111.  No legality check
 * (the reference has none either); `to` must be empty.  winner[i] in {0,1,2}. */
int ccx_apply(ccx_handle *h, int64_t n, uint64_t *state, const uint8_t *from, const uint8_t *to,
              uint8_t *winner);

/* out[i*5 + {0..4}] = check_win, player_progress(1), player_progress(2), player_forward_distance(1),
 * player_forward_distance(2) — board.py:89-111, 254-266, 270-288 */
int ccx_info(ccx_handle *h, int64_t n, const uint64_t *state, int16_t *out);

/* `plies` fused env steps per game: movegen -> selfplay.make_random_move's choice (selfplay.py:93-98:
 * uniform over checkers that can move, then uniform over its destinations) -> place -> check_win; a won
 * game is counted in wins[winner-1] and restarted from Board().  RNG: Philox4x32-10, key = seed,
 * counter = (step0 + t, 0, game id lo, game id hi).  trace (may be NULL): for the first trace_games
 * games and every ply, CCX_TRACE_WORDS words = state words 0-4 before the move, the six destination
 * masks, then from | to<<8 | winner<<16 | checker id<<24; trace[(t*trace_games + g)*12 + k]. */
int ccx_step_random(ccx_handle *h, int64_t n, uint64_t *state, int64_t game_id0, uint64_t seed,
                    uint32_t step0, int32_t plies, uint64_t *wins, uint64_t *trace, int64_t trace_games);

/* GreedyPlayer.decide_move(training=True) — player.py:99-118.  cand_masks[id*n + i] = destinations of
 * checker `id` that are in filtered_best_moves. */
int ccx_greedy_candidates(ccx_handle *h, int64_t n, const uint64_t *state, uint64_t *cand_masks);

/* Game('greedy','greedy').start() — game.py:58-100 — for every game whose status is RUNNING, until it
 * ends (win / repetition stop) or max_plies more plies were played.  Uniform pick among
 * filtered_best_moves (player.py:121) in canonical order with Philox counter (ply, 1, game id).
 * counters (may be NULL): uint64[4] += {plies played, P1 wins, P2 wins, repetition stops}. */
int ccx_play_greedy(ccx_handle *h, int64_t n, uint64_t *state, int64_t game_id0, uint64_t seed,
                    int32_t max_plies, uint64_t *counters);

/* utils.to_model_input(board, side to move) — utils.py:101-160 — written channels-last (n,7,7,7)
 * straight into the network's input tensor; dtype CCX_DTYPE_*. */
int ccx_encode(ccx_handle *h, int64_t n, const uint64_t *state, void *out_nhwc, int dtype);

/* ---- MCTS (MCTS.py:13-153) --------------------------------------------------------------------
 * One tree per root, one simulation at a time per tree (bit-exact visit counts need the reference's
 * strictly sequential order, MCTS.py:121-125; the *_leaves calls below are the opt-in exception).  Selection = PUCT in float64, first maximal edge
 * (MCTS.py:56-69 with the first-choice tie-break); expansion creates every legal edge in canonical
 * order (checker id, then destination cell) with the evaluator's un-normalised prior (MCTS.py:95-109);
 * terminal leaves back up +-1 (MCTS.py:81-90).
 *
 * ccx_mcts_search runs MCTS.search's loop (MCTS.py:121-137) with an in-kernel evaluator:
 *   evaluator 0 = uniform prior 1/294, v = 0.0 (BASELINE configs[3]);
 *   evaluator 1 = deterministic pseudo-random (p, v) keyed by a hash of the to_model_input planes
 *                 (parity-test evaluator, exercises Q-dependent selection and terminal backups).
 * pre_expand = 0: AiPlayer.decide_move (player.py:157-158, unexpanded root, sum N = num_itr - 1);
 * pre_expand = 1: selfplay.make_move (selfplay.py:114-127): root expanded first, then root_noise (may be
 *   NULL; [n][noise_stride] float64, one value per root edge in edge order) is mixed in with weight 0.25.
 * Outputs: visits[n][294] (uint32 N per policy index), pi[n][294] (N^(1/tau) normalised; may be NULL),
 * q[n][294] (root Q; may be NULL), n_nodes[n] (reference node count = edges + 1, or -1 if this tree's
 * edge pool overflowed; may be NULL).  edges_per_tree <= 0 selects 64 * (num_itr + 1). */
int ccx_mcts_search(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t evaluator, int32_t num_itr, double cpuct,
                    double tau, int32_t pre_expand, const double *root_noise, int32_t noise_stride,
                    int32_t edges_per_tree, uint32_t *visits, double *pi, double *q, int32_t *n_nodes);

/* Round-based search for an external evaluator (the policy/value net, model.py:21-24): begin, then per
 * simulation  select -> [ccx_encode + net on leaf_state] -> expand_backup,  finally finalize.
 * leaf_state is uint64[5][n] (state words 0-4 of every tree's leaf; garbage-free for terminal leaves too);
 * p is float64[n][294] soft-maxed policy, v float64[n]; trees whose leaf was terminal ignore them. */
/* min_ply: roots that are not RUNNING or have fewer plies get an inactive tree that every phase skips
 * (self-play opening, selfplay.py:32; finished games); pass -1 to search every root.  n_nodes reports
 * -1 for an overflowed pool and -2 for an inactive tree. */
/* ply_parity: -1 = every root; 0 / 1 = only roots whose ply count is even / odd get an active tree (two-net self-play:
 * model1 moves on even plies, model2 on odd ones, selfplay.py:29,58). */
int ccx_mcts_begin(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t num_itr, int32_t edges_per_tree,
                   int32_t min_ply, int32_t ply_parity);
/* Tree reuse (opt-in): ccx_mcts_begin, except that tree i may start from the subtree the previous search on this handle grew
 * below its new root.  S = num_itr and E = edges_per_tree > 0 ? edges_per_tree : 64 (S + 1) as for ccx_mcts_begin.
 *   Source: tree i continues tree i of the previous search; prev (device int64[n], may be NULL) names another source tree per
 *     tree (a compacted batch), an entry outside [0, trees of the previous search) or -1 means "start fresh".
 *   Match: the node of the source tree at depth 1 or 2 below its root whose state words 0-4 equal roots[.][i] (META's
 *     status byte masked, as the root of every search is stored).
 *   A fresh tree, exactly as ccx_mcts_begin builds it, whenever: the root is inactive (min_ply / ply_parity, then also as
 *     ccx_mcts_begin); no node matches; the match is not expanded; the source tree overflowed or was inactive; the pool was
 *     reallocated since the source search, or the evaluator changed in between (ccx_net_load*, a ccx_net_set_mode that changes
 *     the mode, a ccx_net_set_symmetry that changes the mode or seed — with an external evaluator the caller keeps it the same); or the subtree holds more than carry (S + 2)
 *     nodes, more than carry E edges, or more than carry (S + 1) visits over the new root's edges.
 *   Carry: otherwise the match's subtree becomes tree i, the match its root; per edge N, W, Q, P and the move, each node's
 *     edge order and terminal info are kept bit for bit (node / edge indices are renumbered; no result depends on them).  The
 *     per-search bookkeeping starts over: tie-rule simulation index 0 and root hash of the new root; finalize reports carried
 *     edges + new edges + 1 nodes.  The carried root is expanded, so every selection of the search is a simulation (a one-leaf
 *     search with R rounds adds R visits; leaf-parallel rounds select up to `leaves` leaves from the first round on).
 *     root_noise (may be NULL; [n][noise_stride], noise_normalize as for ccx_mcts_expand_backup) is mixed into a carried root's
 *     priors here; pass the same noise to the rounds, which mix it into the fresh roots they expand.
 *   reused (device int32[n], may be NULL): 1 / 2 = carried from a match at that depth, 0 = fresh, -2 = inactive.
 * The trees' pools hold (1 + carry) times one search's nodes, edges and path, plus a gather scratch of carry times
 * (ccx_mcts_pool_bytes counts both).  carry = 0 makes every tree fresh. */
int ccx_mcts_begin_reuse(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t num_itr, int32_t edges_per_tree,
                         int32_t min_ply, int32_t ply_parity, int32_t carry, const int64_t *prev,
                         const double *root_noise, int32_t noise_stride, int32_t noise_normalize, int32_t *reused);
/* Per-tree search budgets (opt-in; KataGo's playout cap randomization, Wu 2019, arXiv:1902.10565 §3.1): ccx_mcts_begin, except
 * that tree i makes at most b_i = clamp(budget[i], 0, num_itr) selections in this search (budget: device int32[n], read once
 * here: later changes to it do not affect the running search).  The root expansion is the first selection.  Per round, a tree
 * that has made b_i selections is skipped by every phase like an inactive tree, without being flagged: ccx_mcts_select writes
 * the start position into its leaf_state column, ccx_mcts_expand_backup ignores its p / v, ccx_mcts_run_net does the same in
 * its fused rounds, and ccx_mcts_finalize reports the tree as its selections left it.  root_noise of ccx_mcts_expand_backup /
 * ccx_mcts_run_net is mixed only into trees with b_i == num_itr (a full search); a shorter one gets none.  So tree i ends bit
 * for bit (visits, Q, node count; either tie rule, whose simulation index is the tree's own) like the same root searched
 * without budget for num_itr rounds with the same noise (b_i == num_itr), or for b_i rounds without noise (b_i < num_itr).
 * Every net mode and symmetry mode applies.  The budget holds until the next begin; budgeted trees refuse with
 * CCX_ERR_UNSUPPORTED the Gumbel mode (also at this begin) and leaf-parallel calls with leaves > 1.  ccx_mcts_search,
 * ccx_mcts_begin and ccx_mcts_begin_reuse start searches without budgets; a reuse begin carries nothing from budgeted trees
 * (every tree starts fresh).  ccx_mcts_run_net on budgeted trees compacts the net batch: in each round only the
 * trees whose selection reached a leaf to evaluate take net rows (R adjacent rows each, R = 2 with the symmetry mean), packed
 * from the first row of the batch (of each half when the batch is split over two streams) in arbitrary order; a device counter
 * holds the row count and the net kernels evaluate only those rows. */
int ccx_mcts_begin_budget(ccx_handle *h, int64_t n, const uint64_t *roots, int32_t num_itr, int32_t edges_per_tree,
                          int32_t min_ply, int32_t ply_parity, const int32_t *budget);
/* PUCT tie rule of this handle's searches (MCTS.py:65-72).  mode 0 (default): the first maximal edge (what the reference
 * does when `random.choice` is replaced by seq[0]; the bit-exact parity mode).  mode 1: the reference's rule — chosen_edges =
 * the first edge attaining the maximum plus every LATER edge with fabs(QU - max) < EPSILON (1e-5, config.py:36), one of them
 * drawn uniformly — with Philox4x32-10 in place of Python's `random`: key = seed, counter = (simulation index of the tree,
 * depth, tree uid ^ root hash), index = mulhi(x, len(chosen_edges)).  uid of tree i = uid0 + i; root hash = fold32(OCC1 *
 * 0x9E3779B97F4A7C15 + OCC2 * 0xC2B2AE3D27D4EB4F + (META & 0xFFFFFFFFFFFF)): the draws of a search are a function of
 * (seed, uid, root position), never of what the handle searched before. */
int ccx_mcts_set_tiebreak(ccx_handle *h, int32_t mode, uint64_t seed, int64_t uid0);
int ccx_mcts_select(ccx_handle *h, int64_t n, double cpuct, uint64_t *leaf_state);
/* The same rounds with the library's own net as the evaluator (ccx_net_load / ccx_net_load_tc, mode from
 * ccx_net_set_mode), fused: per round  select + to_model_input -> net forward -> float64 softmax + expand +
 * backup  (4 launches, priors never leave the SM).  Equivalent to `rounds` x (ccx_mcts_select, ccx_net_eval,
 * ccx_mcts_expand_backup); root_noise is applied in the first round only (selfplay.py:117-124). */
int ccx_mcts_run_net(ccx_handle *h, int64_t n, int32_t rounds, double cpuct, const double *root_noise, int32_t noise_stride,
                     int32_t noise_normalize);
/* root_noise is applied to trees whose expanded leaf is the root; noise_normalize != 0 divides each
 * tree's first n_edges values by their sum first (raw gamma draws -> Dirichlet, selfplay.py:121). */
int ccx_mcts_expand_backup(ccx_handle *h, int64_t n, const double *p, const double *v, const double *root_noise,
                           int32_t noise_stride, int32_t noise_normalize);
int ccx_mcts_finalize(ccx_handle *h, int64_t n, double tau, uint32_t *visits, double *pi, double *q, int32_t *n_nodes);

/* Leaf-parallel rounds (opt-in; leaves == 1 is exactly the one-leaf call each of these names).  A round selects m leaves per
 * tree one after another: m = 1 while the tree's root is unexpanded, otherwise min(leaves, selections left in this call), so a
 * search makes as many selections as the one-leaf search.  Each pending selection puts one virtual loss on every edge of its
 * path: later descents of the round use N' = N + V, N_sum' = sum N' and Q' = (W - V) / (N + V) (a loss for the player moving
 * along the edge) while N, W, Q stay the real statistics.  A terminal leaf is backed up at once; a leaf node already chosen by a
 * pending selection of the round is a duplicate and is not evaluated.  The backup phase runs the selections in order: a first
 * occurrence is expanded (root_noise mixed in when it is the root), a duplicate reuses its first occurrence's value, and every
 * pending path loses its virtual loss and gets the usual backup.  The tie rule's simulation index counts every selection.
 * Leaf slot (tree i, leaf k) = column i*leaves + k: leaf_state uint64[5][n*leaves], p float64[n*leaves][294],
 * v float64[n*leaves]; a slot with nothing to evaluate holds the start position and its output is ignored.
 * leaves: 1..CCX_MAX_LEAVES.  The per-leaf storage (paths, leaf records, a virtual-loss count per edge) is allocated on the first
 * call with leaves > 1 and counted in ccx_mcts_pool_bytes. */
#define CCX_MAX_LEAVES 16
/* selections the following ccx_mcts_select_leaves rounds of trees [0, n) may make in all (the "call" of the rule above) */
int ccx_mcts_leaf_budget(ccx_handle *h, int64_t n, int32_t leaves, int32_t sims);
int ccx_mcts_select_leaves(ccx_handle *h, int64_t n, int32_t leaves, double cpuct, uint64_t *leaf_state);
int ccx_mcts_expand_backup_leaves(ccx_handle *h, int64_t n, int32_t leaves, const double *p, const double *v,
                                  const double *root_noise, int32_t noise_stride, int32_t noise_normalize);
/* ccx_mcts_run_net with `sims` selections in rounds of up to `leaves` leaves per tree (1 + ceil((sims - 1) / leaves) rounds);
 * net batch n*leaves; the same results as the three calls above with the net as the evaluator */
int ccx_mcts_run_net_leaves(ccx_handle *h, int64_t n, int32_t sims, int32_t leaves, double cpuct, const double *root_noise,
                            int32_t noise_stride, int32_t noise_normalize);
/* Root edge list of every tree in edge order (Edge.stats of root.edges, MCTS.py:24-37): n_edges[n], and per
 * edge j < min(n_edges, stride): moves = checker id << 8 | destination cell, N, W, P ([n][stride] each).
 * ccx_mcts_set_root_priors overwrites P (callers mix Dirichlet noise into it, selfplay.py:121-124). */
int ccx_mcts_get_root(ccx_handle *h, int64_t n, int32_t stride, int32_t *n_edges, uint16_t *moves, uint32_t *N, double *W,
                      double *P);
int ccx_mcts_set_root_priors(ccx_handle *h, int64_t n, int32_t stride, const double *P);
int64_t ccx_mcts_pool_bytes(const ccx_handle *h);

/* Gumbel search (opt-in; Danihelka et al., ICLR 2022; mctx gumbel_muzero_policy with qtransform_completed_by_mix_value).
 * enabled != 0 switches this handle's searches to it until a call with enabled = 0.  In the mode ccx_mcts_begin, ccx_mcts_select,
 * ccx_mcts_expand_backup and ccx_mcts_run_net run one leaf per round under the Gumbel rules (root_noise must be NULL); a search
 * begun with num_itr = R makes R rounds, the first of which expands the root, so S = R - 1 simulations follow it; finish it
 * with ccx_mcts_finalize_gumbel.  ccx_mcts_search, ccx_mcts_begin_reuse, ccx_mcts_select_leaves and ccx_mcts_run_net_leaves
 * (leaves > 1) return CCX_ERR_UNSUPPORTED in the mode.  Per tree, logit(a) = log(max(P(a), DBL_MIN)) over the node's edges:
 *   root expansion: g(a) = scale * Gumbel(0, 1) per edge (Philox4x32-10, key (seed lo, uid lo), counter (root hash, edge index,
 *     uid hi, seed hi); uid and root hash as for the tie rule, so slot ids key the draws), m' = min(considered, edges);
 *   root simulation k: among the edges whose N equals mctx's get_sequence_of_considered_visits(m', S)[k], the arg-max of
 *     max(-1e9, g + (logit - max logit) + sigma);
 *   other nodes: the arg-max of pi'(a) - N(a) / (1 + sum N), pi' = softmax(logit + sigma);
 *   sigma = (c_visit + max N) * c_scale * (q - min q) / max(max q - min q, 1e-8) over the node's edges, q = the edge's Q if
 *     visited, else (v + sum N * sum_visited(p Q) / sum_visited(p)) / (1 + sum N), p = softmax(logit) floored at DBL_MIN and
 *     v the evaluator's value of the node (v alone while no edge is visited).
 * Arg-maxes take the first maximal edge (no tie rule); terminal leaves back up +-1 as in PUCT.  The per-node values, root draws
 * and the schedule table are allocated by the first begin in the mode, freed with the trees, and counted in
 * ccx_mcts_pool_bytes.  considered >= 1, scale >= 0, c_visit >= 0, c_scale >= 0. */
int ccx_mcts_set_gumbel(ccx_handle *h, int32_t enabled, int32_t considered, double scale, double c_visit, double c_scale,
                        uint64_t seed);
/* visits, q (may be NULL) and n_nodes (may be NULL) as ccx_mcts_finalize; pi (may be NULL) float64[n][294] = the improved
 * policy softmax(logit + sigma) over the root's edges, 0 elsewhere; action (may be NULL) int32[n] = the root's arg-max of the
 * score above with considered visit = max N; an inactive, overflowed or unexpanded tree gets action -1 and pi 0. */
int ccx_mcts_finalize_gumbel(ccx_handle *h, int64_t n, uint32_t *visits, double *pi, double *q, int32_t *action, int32_t *n_nodes);

/* ---- policy/value net (model.py:15-145) -----------------------------------------------------------
 * ccx_net_load takes the BN-folded fp32 weights packed by chinesecheckersagent_b200/model.py (layout in
 * csrc/ccx_net.cu; ccx_net_num_weights() floats, HOST pointer — the one non-_host function that reads
 * host memory, like Model.load_weights reading a file, model.py:45-47).
 * ccx_net_forward: Keras predict on a batch: planes (n,7,7,7) channels-last of dtype CCX_DTYPE_* ->
 *   logits float32[n][294] (linear policy head, model.py:112-116) and value float32[n] (tanh, :98-103).
 * ccx_softmax_f64: utils.softmax in float64 over all 294 logits (model.py:23, utils.py:187-192);
 *   v (may be NULL) receives value widened to float64.
 * ccx_net_eval = utils.to_model_input + Model.predict for packed leaf states (uint64[5][n]): the
 *   evaluator of the round-based MCTS (MCTS.py:93). */
int ccx_net_num_weights(void);
int ccx_net_load(ccx_handle *h, const float *packed_host, int64_t count);
int ccx_net_forward(ccx_handle *h, int64_t n, const void *planes, int dtype, float *logits, float *value);
int ccx_softmax_f64(ccx_handle *h, int64_t n, const float *logits, const float *value, double *p, double *v);
int ccx_net_eval(ccx_handle *h, int64_t n, const uint64_t *leaf_state, double *p, double *v);
/* Tensor-core path (tcgen05.mma, accumulators / residual / 1x1-conv operands in TMEM, the 3x3 conv's operand in shared
 * memory): the weights arrive as a 16-bit operand blob already arranged in the UMMA K-major operand layout — every
 * trunk matrix transposed [N][K + 16] with the layer's bias split over two of the extra columns — plus an fp32 blob
 * (biases again, for the policy dense kernel, and the value-head dense); model.py pack_weights_tc builds both, sizes
 * from ccx_net_tc_blob_bytes / ccx_net_tc_num_floats; HOST pointers.
 * ccx_net_forward_tc takes uint8 planes (n,7,7,7).  ccx_net_set_mode(1) makes ccx_net_eval use it. */
int ccx_net_tc_blob_bytes(void);
int ccx_net_tc_num_floats(void);
/* fp16 = 0: the blob holds bf16 operands (kind::f16 with BF16 formats); fp16 = 1: IEEE half operands */
int ccx_net_load_tc(ccx_handle *h, const void *bf16_blob_host, int64_t blob_bytes, const float *f32_host, int64_t n_floats,
                    int32_t fp16);
int ccx_net_forward_tc(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value);
int ccx_net_set_mode(ccx_handle *h, int32_t mode);
/* Mirror-symmetric net evaluation (opt-in), a property of the handle's net evaluator like ccx_net_set_mode.  The game is
 * symmetric under the mirror cell (r, c) -> (6 - c, 6 - r): to_model_input of the mirrored position is the planes mirrored so,
 * and policy index a = id*49 + r*7 + c maps to mirror(a) = id*49 + (6-c)*7 + (6-r).  Modes:
 *   0 (default): one evaluation as is, bit for bit what the handle does without this call.
 *   1, random: position s is evaluated mirrored when bit 0 of the first word of Philox4x32-10 with key (seed lo, seed hi) and
 *     counter (h(s), 0x53594D, 0, 0) is 1; h(s) = fold32(OCC1 * 0x9E3779B97F4A7C15 + OCC2 * 0xC2B2AE3D27D4EB4F +
 *     (META & 0xFFFFFFFFFFFF)), the tie rule's root hash applied to s, so s gets the same orientation wherever it is evaluated.
 *     Mirrored: p[a] = softmax(logits(mirrored planes))[mirror(a)] and v = the value of the mirrored planes.
 *   2, mean: p[a] = (p_id[a] + p_mir[mirror(a)]) * 0.5 and v = ((double)v_id + (double)v_mir) * 0.5 (round-to-nearest adds, the
 *     multiply is exact); the net evaluates two rows per position (the batch doubles).
 * Each p is ccx_softmax_f64's float64 softmax over all 294 logits.  It applies to ccx_net_eval and to the fused loops
 * (ccx_mcts_run_net, ccx_mcts_run_net_leaves, in the PUCT and the Gumbel modes), which compute the same bits as the round trips
 * with ccx_net_eval.  ccx_net_forward*, ccx_softmax_f64 and the in-kernel evaluators of ccx_mcts_search are unaffected.  A
 * change of mode or seed invalidates the cached round graph and the trees a reuse begin could carry.  mode outside 0..2:
 * CCX_ERR_ARG. */
int ccx_net_set_symmetry(ccx_handle *h, int32_t mode, uint64_t seed);
/* Accurate tensor-core mode (ccx_net_set_mode(h, 2); needs ccx_net_load, ccx_net_load_tc and ccx_net_load_acc): every product
 * in split precision, a_hi*w_hi + a_lo*w_hi + a_hi*w_lo with IEEE-half terms and fp32 accumulation, policy dense layer
 * included — the tensor-core path at the fp32 restatement's accuracy (|dp|, |dv| << 1e-3).  The blob (model.py pack_weights_acc):
 * per matrix [hi: N x (K+16), bias columns][lo: N x K] in the UMMA operand layout; HOST pointer. */
/* forward pass of uint8 planes (n,7,7,7) in the mode selected by ccx_net_set_mode (0 fp32 SIMT, 1 tensor core, 2 accurate) */
int ccx_net_forward_u8(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value);
int ccx_net_acc_blob_bytes(void);
int ccx_net_load_acc(ccx_handle *h, const void *blob_host, int64_t blob_bytes);
/* Tiles in flight per CTA of the accurate trunk kernel: 1-3 = k_net_trunk_accm (one CTA per SM, that many 256-thread contexts
 * sharing the streamed weight slots), 0 = k_net_trunk_acc (one tile per CTA, two CTAs per SM), -1 = automatic (the default: the
 * environment variable CCX_ACC_CTX if set, else as many contexts, up to 3, as the batch has tiles per SM).  Every setting computes
 * the same bits (model.py:58-145 has no notion of it): it exists for A/B timing and tests. */
int ccx_net_set_acc_contexts(ccx_handle *h, int32_t contexts);

/* ---- self-play (selfplay.py:11-133) and trajectory packing (utils.py:60-73) -------------------------
 * One game slot per tree, all slots advanced one ply per iteration; see chinesecheckersagent_b200/selfplay.py
 * for the driver loop.  Records live in caller-owned device buffers indexed rec = iter*n + slot:
 *   rec_state uint64[rec_iters*n][5], rec_visits uint16[rec_iters*n][294], rec_flag uint8[rec_iters*n]
 *   (low nibble: 0 none, 1 pending, 2 mover won, 3 mover lost, 4 dropped; 0x10 = pi uses DET_TREE_TAU).
 *   The buffers are a RING over iterations: the record of (iter, slot) lives at row (iter % rec_iters)*n + slot, so a caller
 *   that consumes finished records in time (chinesecheckersagent_b200/selfplay.py does) can play indefinitely.
 * counters uint64[8] += {plies, P1 wins, P2 wins, repetition discards, progress-limit discards,
 *   overflow discards (edge pool or record ring; status CCX_ST_OVERFLOW), records kept, games kept}.
 * ccx_gamma_noise: raw Gamma(alpha) draws [n][stride] for the root Dirichlet noise (selfplay.py:121).
 * ccx_selfplay_advance: opening plies (ply < random_plies) take selfplay.make_random_move's choice
 *   (selfplay.py:83-104); later plies sample np.random.choice(294, p=pi) from this iteration's visit counts
 *   (MCTS.py:131-140, tau = 0.01 once recorded + random_plies > tau_switch, selfplay.py:62-65), record
 *   (state, visits) (selfplay.py:128), then apply the move and the repetition / progress / win / useless-move
 *   rules in the reference's order (selfplay.py:40-74).  Game uid = serial*total_slots + uid0 + slot keys Philox.
 * ccx_selfplay_finish: labels the records of games that ended (reward from the mover's point of view,
 *   utils.py:65-71) or drops them for discarded games (selfplay.py:47,74); a running game that has been recorded for
 *   max_game_iters iterations (> 0) is discarded as CCX_ST_OVERFLOW before its records wrap around the ring.
 *   restart != 0 resets the slot of an ended game — if starts_left (device int64, may be NULL) is NULL or still positive:
 *   train.py:58-64 plays exactly num_self_play games, so the caller sets starts_left = num_self_play - n and drains.  The
 *   slots that ended in one iteration take the remaining starts in slot order (deterministic), *starts_left is decremented
 *   by the number of restarts.  A slot that may not restart keeps its final status.
 * ccx_traj_pack: gathers kept records rows[m] into out_state uint64[5][m] (feed to ccx_encode for board_x),
 *   pi_y float32[m][294] and v_y int8[m]. */
int ccx_gamma_noise(ccx_handle *h, int64_t n, int32_t stride, double alpha, uint64_t seed, uint32_t iter, int64_t uid0,
                    double *out);
/* Slot identities for a COMPACTED batch.  By default slot / tree i of a call is identified as uid0 + i wherever a Philox stream is
 * keyed by it (ccx_gamma_noise, ccx_selfplay_advance, the tie rule of the searches).  With slot_ids != NULL (device int64[n], stays
 * referenced until reset with NULL) entry i is identified as slot_ids[i] instead, so a caller can drop finished slots from the batch
 * (chinesecheckersagent_b200/selfplay.py: BatchedSelfPlay.compact) and the surviving games continue bit for bit as they would have. */
int ccx_set_slot_ids(ccx_handle *h, const int64_t *slot_ids);
int ccx_selfplay_advance(ccx_handle *h, int64_t n, uint64_t *state, const uint32_t *visits, const int32_t *tree_nodes,
                         uint64_t seed, int32_t iter, int64_t uid0, const int64_t *serial, int64_t total_slots,
                         int32_t random_plies, int32_t tau_switch, int32_t move_limit, uint64_t *rec_state,
                         uint16_t *rec_visits, uint8_t *rec_flag, int32_t rec_iters, uint64_t *counters,
                         uint32_t *move_log /* may be NULL: [rec_iters*n] from | to<<8 | status<<16 | 1<<24 | mcts<<25 */);
int ccx_selfplay_finish(ccx_handle *h, int64_t n, uint64_t *state, int32_t iter, int32_t *start_iter, int64_t *serial,
                        const uint64_t *rec_state, uint8_t *rec_flag, int32_t rec_iters, int32_t max_game_iters, int32_t restart,
                        int64_t *starts_left, uint64_t *counters);
int ccx_traj_pack(ccx_handle *h, int64_t m, const int64_t *rows, const uint64_t *rec_state, const uint16_t *rec_visits,
                  const uint8_t *rec_flag, uint64_t *out_state, float *pi_y, int8_t *v_y);
/* Policy targets other than visit counts (the Gumbel search's improved policy): ccx_selfplay_record_pi stores pi float64[n][294]
 * as float32 row (iter % rec_iters) * n + slot of rec_pi, for the slots whose pi row is not all zero (the searched ones, which
 * ccx_selfplay_advance records in the same row); ccx_traj_pack_pi is ccx_traj_pack with pi_y copied from rec_pi. */
int ccx_selfplay_record_pi(ccx_handle *h, int64_t n, int32_t iter, const double *pi, float *rec_pi, int32_t rec_iters);
int ccx_traj_pack_pi(ccx_handle *h, int64_t m, const int64_t *rows, const uint64_t *rec_state, const float *rec_pi,
                     const uint8_t *rec_flag, uint64_t *out_state, float *pi_y, int8_t *v_y);

/* ---- self-play resignation (opt-in; AlphaZero's resignation with no-resign probe games) -----------------------------------
 * Resign value of one search.  Tree i (this handle's tree pool, slot i) after the search's last round, root edges in edge order,
 * N the edge's visits and Q = W / N (0 for N = 0), exactly as ccx_mcts_finalize reports them:
 *   v_root = sum N*Q / sum N,  q_best = Q of the first edge with the maximal N,  r = max(v_root, q_best)
 * (the root value and the best child's value, both from the view of the player to move).  Both sums are float64 in warp order:
 * lane l sums N*Q (resp. N) of edges l + 32c for c = 0..3 (0.0 past the last edge), then an xor butterfly over 16, 8, 4, 2, 1.
 * A root with sum N = 0, or a tree that is inactive or overflowed, has no value.  The rule is the same in every search mode
 * (PUCT, leaf-parallel rounds, Gumbel, symmetric evaluation); with tree reuse the carried visits are part of the root.
 * Streak.  Each player of each game keeps its count of consecutive searched plies with r < threshold (a ply with
 * r >= threshold resets it).  When it reaches `plies` (1..8) the player resigns: status CCX_ST_RESIGN_WON_P1 / _P2 (the other
 * player wins), no move is played, the position is not recorded.  threshold <= -1 never resigns (r >= -1): track-only.
 * Probe games.  At its start a game is a probe when u < probe, u = x / 2^32, x = the first word of Philox4x32-10 with key
 * (seed lo, seed hi) and counter (slot id lo, slot id hi, serial lo, 0x52534750); slot id = slot_ids[i] (ccx_set_slot_ids) or
 * uid0 + i, serial = the slot's game serial.  A probe never resigns; the first time its streak reaches `plies` the player who
 * would have resigned is remembered.
 * Window.  Over a player's searched plies, the minimum of max(r over its last `plies` searched plies) (windows of `plies`
 * values only; +inf while it has fewer): the largest threshold at which that player would not have resigned is exactly it.
 * resign_state: int64[n][CCX_RESIGN_WORDS], caller-owned, every entry of word 0 = -1 before first use.  It belongs to the game
 * whose serial is in word 0; a slot whose serial changed (a restart) starts clean.  Other words are the kernels' business.
 * counters uint64[6] += {games resigned, probe games, probe games with a would-resign, false positives, samples written,
 * samples dropped}; probe games count once they end with a winner (discarded games are left out of every count).
 *
 * ccx_selfplay_resign: between the search and ccx_selfplay_advance, one warp per slot: r of every tree with a value, streak and
 *   window update, resignation.  value_out (may be NULL) float64[n] = r, NaN where no value.  With two nets, call it on each
 *   net's handle after its search: each handle sees the active trees of its own parity.
 * ccx_selfplay_resign_account: between ccx_selfplay_advance and ccx_selfplay_finish, for the games that ended in this iteration
 *   (a status other than RUNNING and start_iter <= iter, the games ccx_selfplay_finish settles next): a probe game won by a player
 *   counts a probe game, a would-resign and, when the would-be resigner won, a false positive.  A game that resignation could not
 *   have cut short (a probe, or any game when threshold <= -1) and that has a winner appends the winner's window value to
 *   samples[sample_cap] (device float64; written in slot order after the samples of earlier calls; past sample_cap: dropped).
 * ccx_selfplay_finish labels a resigned game's records like a win of the player who did not resign and counts it as that win. */
#define CCX_RESIGN_WORDS 20
#define CCX_RESIGN_MAX_PLIES 8
int ccx_selfplay_resign(ccx_handle *h, int64_t n, uint64_t *state, uint64_t seed, int64_t uid0, const int64_t *serial,
                        double threshold, int32_t plies, double probe, int64_t *resign_state, double *value_out, uint64_t *counters);
int ccx_selfplay_resign_account(ccx_handle *h, int64_t n, const uint64_t *state, int32_t iter, const int32_t *start_iter,
                                const int64_t *serial, uint64_t seed, int64_t uid0, double threshold, double probe,
                                int64_t *resign_state, uint64_t *counters, double *samples, int64_t sample_cap);

/* ---- self-play playout cap randomization (opt-in; KataGo, Wu 2019, arXiv:1902.10565 §3.1) --------------------------------
 * Before each iteration's search, one thread per slot writes the slot's budget for ccx_mcts_begin_budget: full_budget when
 * x / 2^32 < p, fast_budget otherwise, x = the first word of Philox4x32-10 with key (seed lo, seed hi) and counter (slot id lo,
 * slot id hi, serial lo, 0x50430000 + ply); slot id = slot_ids[i] (ccx_set_slot_ids) or uid0 + i, serial = the slot's game
 * serial, ply = the game's ply count.  The draw is a function of the game and the ply: batch compaction changes nothing.  The
 * counter word never equals the resignation probe's (0x52534750).  A slot that searches this iteration (RUNNING and
 * ply >= min_ply) adds 1 to counters[0] (full) or counters[1] (fast); the others get full_budget, which no search reads.
 * keep (device uint8[n], may be NULL) = 0 for a slot that makes a fast search this iteration, else 1.  A full search keeps the
 * root noise (its budget is the begin's num_itr); the caller clears the record flag of every slot with keep = 0 between
 * ccx_selfplay_advance and ccx_selfplay_finish, so only full searches become policy targets (with fast_budget == full_budget
 * the two kinds search alike, noise included, and still only the full draws are kept).  p in [0, 1],
 * 0 <= fast_budget <= full_budget, else CCX_ERR_ARG. */
int ccx_selfplay_playout_cap(ccx_handle *h, int64_t n, const uint64_t *state, uint64_t seed, int64_t uid0, const int64_t *serial,
                             int32_t min_ply, double p, int32_t full_budget, int32_t fast_budget, int32_t *budget, uint64_t *counters,
                             uint8_t *keep);

/* Self-test of the tcgen05/TMEM plumbing used by the bf16 net kernel: D[128][N] = A[128][K] * Bt[N][K]^T
 * (bf16 in, fp32 out; K multiple of 16 up to 512, N multiple of 16 up to 64).  Used by the GPU tests. */
int ccx_debug_umma_gemm(ccx_handle *h, const void *A, const void *Bt, int32_t K, int32_t N, float *D);
/* same, with A [rows x K] held in the row-contiguous operand layout of the 3x3 conv and the descriptor start moved by
 * `shift` rows: D[128 x N] = A[shift .. shift+127] * Bt^T (self-test of 16-byte-granular descriptor starts). */
/* same with the A operand [128 x 64] read from TMEM (tcgen05.mma "ts" form; packed pairs written with tcgen05.st) */
int ccx_debug_umma_gemm_ts(ccx_handle *h, const void *A, const void *Bt, int32_t N, float *D);
int ccx_debug_umma_gemm_rows(ccx_handle *h, const void *A, int32_t rows, int32_t shift, const void *Bt, int32_t K, int32_t N,
                             float *D);

/* ---- arena / evaluation games (game.py:58-100; ai_vs_ai.py:28-52; ai_vs_greedy.py:26-59; train.py:150-231) ----
 * One Game.start ply for every RUNNING game.  visits != NULL: the mover is an AiPlayer whose MCTS result this is
 * (uint32[n][294] from ccx_mcts_finalize, tree_nodes its n_nodes): the move is sampled from N^(1/tau), tau switching
 * to DET_TREE_TAU once more than tau0_after plies were played (player.py:151-154).  visits == NULL: the mover is the
 * GreedyPlayer (uniform among filtered_best_moves).  Then winner / repetition stop / optional move limit
 * (move_limit = 0: off).  A search whose edge pool overflowed stops the game with CCX_ST_OVERFLOW.
 * counters uint64[4] += {plies, P1 wins, P2 wins, stopped games}. */
int ccx_game_advance(ccx_handle *h, int64_t n, uint64_t *state, const uint32_t *visits, const int32_t *tree_nodes, uint64_t seed,
                     int64_t uid0, double tau, int32_t tau0_after, int32_t move_limit, uint64_t *counters);

/* ---- greedy supervised-data generator (data_generators.py:14-80; train_on_greedy.py:17-42) ---------------
 * Batched GreedyDataGenerator.generate_play: every game starts from state[.][i] (ccx_reset: start position or
 * randomised), optionally plays `random_plies` random legal plies (random_start), then both sides play
 * GreedyPlayer.decide_move(training=True) with a uniform pick among filtered_best_moves until a win.  Every
 * position is a record (state words 0-4, candidate masks); records of randomised games lose their first
 * `drop_first` entries (data_generators.py:74-75).  The reference's 0.1 s "stuck" limit is a ply count here:
 * a game that reaches `stuck_plies` records keeps its first `stuck_keep` with reward 0 (data_generators.py:65-67).
 * Two passes: offsets == NULL counts (n_records[n], winner[n] out); then with offsets = exclusive prefix sum of
 * n_records and total_records = their sum, the same call writes rec_state uint64[5][M], rec_cand uint64[6][M],
 * rec_v int8[M] (+1/-1/0 from the side to move's point of view, utils.py:65-71) and optionally rec_game int32[M].
 * ccx_cand_to_pi turns candidate masks into pi_y float32[M][294] (uniform over the candidates, :45-51). */
int ccx_greedy_generate(ccx_handle *h, int64_t n, const uint64_t *state, int64_t game_id0, uint64_t seed, int32_t random_plies,
                        int32_t drop_first, int32_t stuck_plies, int32_t stuck_keep, int32_t *n_records, uint8_t *winner,
                        const int64_t *offsets, int64_t total_records, uint64_t *rec_state, uint64_t *rec_cand, int8_t *rec_v,
                        int32_t *rec_game);
int ccx_cand_to_pi(ccx_handle *h, int64_t m, const uint64_t *rec_cand, float *pi_y);

/* ---- host-buffer variants: the reference-facing path with H2D/D2H inside the call -------------- */
int ccx_movegen_host(ccx_handle *h, int64_t n, const uint64_t *state_host, uint64_t *dest_masks_host);
int ccx_apply_host(ccx_handle *h, int64_t n, uint64_t *state_host, const uint8_t *from_host,
                   const uint8_t *to_host, uint8_t *winner_host);
int ccx_step_random_host(ccx_handle *h, int64_t n, uint64_t *state_host, int64_t game_id0, uint64_t seed,
                         uint32_t step0, int32_t plies, uint64_t *wins_host);
int ccx_encode_host(ccx_handle *h, int64_t n, const uint64_t *state_host, void *out_host, int dtype);
int ccx_info_host(ccx_handle *h, int64_t n, const uint64_t *state_host, int16_t *out_host);
int ccx_greedy_candidates_host(ccx_handle *h, int64_t n, const uint64_t *state_host, uint64_t *cand_masks_host);

#ifdef __cplusplus
}
#endif
#endif /* CCX_H */
