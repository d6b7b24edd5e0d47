/*
 * leaves_oracle.c — CPU restatement of the engine's leaf-parallel MCTS (leaves_per_round > 1; include/ccx.h
 * ccx_mcts_*_leaves).  TEST INFRASTRUCTURE, NOT PRODUCT: built by leaves_oracle.py together with the one-leaf oracle's
 * sources (oracle/ccx_oracle*.c, for the board, encoding, Philox and thread-pool routines) into its own library.
 *
 * Same conventions as oracle/ccx_oracle_mcts.c: the reference's object formulation (eager child nodes, MCTS.py:97-109),
 * canonical edge order (checker id, then destination r*7+c), float64 PUCT without contraction (-ffp-contract=off), the
 * first maximal edge or the engine's tie rule 1 (epsilon-tie list, Philox draw keyed by (seed; simulation index, depth,
 * uid ^ root hash * 0x9E3779B9, (uid >> 32) ^ 0x7E1B)), and the two test evaluators (uniform 1/294, v = 0; planes hash).
 */
#include "ccx_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

uint64_t orc_planes_hash(const uint8_t planes[7][7][7]);        /* oracle/ccx_oracle_mcts.c */

typedef struct { int on; uint64_t seed, uid; uint32_t serial, sim; } tie_rule;

static int cmp_dest(const void *a, const void *b)
{
    const int8_t *x = (const int8_t *)a, *y = (const int8_t *)b;
    return (x[0] * 7 + x[1]) - (y[0] * 7 + y[1]);
}

static void eval_uniform(void *ctx, const uint8_t planes[7][7][7], double p[ORC_NACT], double *v)
{
    (void)ctx; (void)planes;
    for (int i = 0; i < ORC_NACT; i++) p[i] = 1 / 294.;
    *v = 0.0;
}

/* P[i] = philox(H, (i,7,0,0)).x / 2^32; v = philox(H, (294,7,0,0)).x / 2^31 - 1, H = orc_planes_hash(planes) */
static void eval_hash(void *ctx, const uint8_t planes[7][7][7], double p[ORC_NACT], double *v)
{
    (void)ctx;
    uint64_t h = orc_planes_hash(planes);
    uint32_t out[4];
    for (int i = 0; i < ORC_NACT; i++) {
        orc_philox((uint32_t)h, (uint32_t)(h >> 32), (uint32_t)i, 7u, 0u, 0u, out);
        p[i] = (double)out[0] / 4294967296.0;
    }
    orc_philox((uint32_t)h, (uint32_t)(h >> 32), 294u, 7u, 0u, 0u, out);
    *v = (double)out[0] / 2147483648.0 - 1.0;
}

/* A round makes m selections: m = 1 while the root is unexpanded, else min(L, selections left).  Selection k runs the
 * PUCT descent (MCTS.py:56-69) on effective statistics: V(e) = pending selections of this round through e, N' = N + V,
 * N_sum' = sum N', Q' = (W - V) / (N + V) when V > 0 (a loss for the player moving along e), else Q.  A terminal leaf is
 * backed up at once; a leaf node already chosen by a pending selection of this round is a duplicate (not evaluated, no
 * expansion).  Then, k in order: a first occurrence is evaluated and expanded, a duplicate takes its first occurrence's
 * value, and each pending path drops one virtual loss per edge and gets the usual backup.  Own node/edge types and own
 * expansion, independent of the one-leaf oracle it is compared with. */
typedef struct vnode vnode;
typedef struct {
    int in_player;
    int idx;
    int64_t N, V;             /* V: virtual losses, an integer count kept beside the edge, never folded into W */
    double W, Q, P;
    vnode *out;
} vedge;

struct vnode {
    orc_board state;
    int player, n_edges, visited;
    vedge *edges;
};

typedef struct { vnode **all; int n, cap; } varena;

static vnode *vnew_node(varena *a, const orc_board *b, int player)
{
    vnode *nd = (vnode *)calloc(1, sizeof(vnode));
    nd->state = *b; nd->player = player;
    if (a->n == a->cap) { a->cap = a->cap ? a->cap * 2 : 1024; a->all = (vnode **)realloc(a->all, sizeof(vnode *) * (size_t)a->cap); }
    a->all[a->n++] = nd;
    return nd;
}

static vnode *vmove_to_leaf(vnode *root, double cpuct, vedge **crumbs, int *ncrumbs, const tie_rule *tie)
{
    vnode *cur = root;
    *ncrumbs = 0;
    int depth = 0;
    while (cur->n_edges != 0) {
        double maxQU = -INFINITY;
        int64_t N_sum = 0;
        vedge *chosen = NULL;
        vedge *list[128]; int nlist = 0;
        for (int i = 0; i < cur->n_edges; i++) N_sum += cur->edges[i].N + cur->edges[i].V;
        for (int i = 0; i < cur->n_edges; i++) {
            vedge *e = &cur->edges[i];
            int64_t Ne = e->N + e->V;
            double Q = e->V > 0 ? (e->W - (double)e->V) / (double)Ne : e->Q;
            double U = cpuct * e->P * sqrt((double)N_sum) / (1. + (double)Ne);
            double QU = Q + U;
            if (QU > maxQU) { maxQU = QU; chosen = e; nlist = 0; list[nlist++] = e; }
            else if (fabs(QU - maxQU) < 1e-5 && nlist < 128) list[nlist++] = e;
        }
        if (tie && tie->on && nlist > 1) {
            uint32_t out[4];
            orc_philox((uint32_t)tie->seed, (uint32_t)(tie->seed >> 32), tie->sim, (uint32_t)depth,
                       (uint32_t)tie->uid ^ (tie->serial * 0x9E3779B9u), (uint32_t)(tie->uid >> 32) ^ 0x7E1Bu, out);
            chosen = list[(uint32_t)(((uint64_t)out[0] * (uint64_t)nlist) >> 32)];
        }
        crumbs[(*ncrumbs)++] = chosen;
        cur = chosen->out;
        depth++;
    }
    return cur;
}

static double vexpand(varena *a, vnode *leaf, orc_eval_fn eval, void *ctx)
{
    uint8_t planes[7][7][7];
    double p[ORC_NACT], v = 0.0;
    orc_to_model_input(&leaf->state, leaf->player, planes);
    eval(ctx, planes, p, &v);
    int8_t mv[6][ORC_MAX_DESTS][2]; int32_t cnt[6];
    orc_get_valid_moves(&leaf->state, leaf->player, mv, cnt);
    int total = 0;
    for (int id = 0; id < 6; id++) total += cnt[id];
    leaf->edges = (vedge *)calloc((size_t)(total ? total : 1), sizeof(vedge));
    for (int id = 0; id < 6; id++) {
        qsort(mv[id], (size_t)cnt[id], 2, cmp_dest);
        int fr = leaf->state.pos[leaf->player - 1][id][0], fc = leaf->state.pos[leaf->player - 1][id][1];
        for (int k = 0; k < cnt[id]; k++) {
            vedge *e = &leaf->edges[leaf->n_edges++];
            int tr = mv[id][k][0], tc = mv[id][k][1];
            orc_board next = leaf->state;
            orc_place(&next, leaf->player, fr, fc, tr, tc);
            e->in_player = leaf->player;
            e->idx = id * 49 + tr * 7 + tc;
            e->P = p[e->idx];
            e->out = vnew_node(a, &next, 3 - leaf->player);
        }
    }
    return v;
}

/* backup of a finished selection: terminal (+-1 from the winner's side) or value v; drop_vl removes its virtual loss */
static void vbackup(vedge **crumbs, int ncrumbs, const vnode *leaf, double v, int terminal, int drop_vl)
{
    for (int i = 0; i < ncrumbs; i++) {
        vedge *e = crumbs[i];
        int same = e->in_player == leaf->player;
        if (drop_vl) e->V -= 1;
        e->N += 1;
        e->W += terminal ? 1.0 * (same ? -1 : 1) : v * (same ? 1 : -1);
        e->Q = e->W / (double)e->N;
    }
}

#define ORC_MAX_LEAVES 16

static void mcts_search_leaves(const uint64_t rootw[8], int32_t num_itr, double cpuct, double tau, int pre_expand, int leaves,
                               const double *root_noise, orc_eval_fn eval, uint32_t visits[ORC_NACT], double pi[ORC_NACT],
                               int32_t *n_nodes, double *q_out, tie_rule *tie, int32_t *visited, int64_t *vl_left)
{
    varena a = {0};
    orc_board b; int tm;
    orc_unpack(rootw, &b, &tm, NULL);
    vnode *root = vnew_node(&a, &b, tm + 1);
    root->visited = 1;
    int nvisited = 1;
    struct { vnode *leaf; vedge **crumbs; int ncrumbs, dup_of; double v; } pend[ORC_MAX_LEAVES];
    for (int k = 0; k < ORC_MAX_LEAVES; k++) pend[k].crumbs = (vedge **)malloc(sizeof(vedge *) * (size_t)(num_itr + 2));
    memset(visits, 0, sizeof(uint32_t) * ORC_NACT);
    memset(pi, 0, sizeof(double) * ORC_NACT);
    if (q_out) memset(q_out, 0, sizeof(double) * ORC_NACT);
    if (pre_expand) {
        if (!orc_check_win(&root->state)) vexpand(&a, root, eval, NULL);
        if (root_noise)
            for (int i = 0; i < root->n_edges; i++) {
                root->edges[i].P *= (1. - 0.25);
                root->edges[i].P += 0.25 * root_noise[i];
            }
    }
    int done = 0;
    while (done < num_itr) {
        int m = root->n_edges == 0 ? 1 : (num_itr - done < leaves ? num_itr - done : leaves);
        int np = 0;
        for (int k = 0; k < m; k++) {                                   /* selections, one after another */
            if (tie) tie->sim = (uint32_t)(done + (pre_expand ? 1 : 0));
            done++;
            int nc;
            vnode *leaf = vmove_to_leaf(root, cpuct, pend[np].crumbs, &nc, tie);
            if (!leaf->visited) { leaf->visited = 1; nvisited++; }
            if (orc_check_win(&leaf->state)) { vbackup(pend[np].crumbs, nc, leaf, 0.0, 1, 0); continue; }
            int dup = -1;
            for (int j = 0; j < np && dup < 0; j++) if (pend[j].leaf == leaf) dup = j;
            pend[np].leaf = leaf; pend[np].ncrumbs = nc; pend[np].dup_of = dup;
            for (int i = 0; i < nc; i++) pend[np].crumbs[i]->V += 1;
            np++;
        }
        for (int j = 0; j < np; j++) {                                  /* backup phase in selection order */
            if (pend[j].dup_of < 0) pend[j].v = vexpand(&a, pend[j].leaf, eval, NULL);
            else pend[j].v = pend[pend[j].dup_of].v;
            vbackup(pend[j].crumbs, pend[j].ncrumbs, pend[j].leaf, pend[j].v, 0, 1);
        }
    }
    double sum = 0.0;
    for (int i = 0; i < root->n_edges; i++) {
        vedge *e = &root->edges[i];
        visits[e->idx] = (uint32_t)e->N;
        pi[e->idx] = pow((double)e->N, 1. / tau);
        if (q_out) q_out[e->idx] = e->Q;
    }
    for (int i = 0; i < ORC_NACT; i++) sum += pi[i];
    if (sum > 0) for (int i = 0; i < ORC_NACT; i++) pi[i] /= sum;
    if (n_nodes) *n_nodes = a.n;
    if (visited) *visited = nvisited;
    int64_t vl = 0;
    for (int i = 0; i < a.n; i++) {
        for (int j = 0; j < a.all[i]->n_edges; j++) vl += a.all[i]->edges[j].V;
        free(a.all[i]->edges); free(a.all[i]);
    }
    if (vl_left) *vl_left = vl;
    free(a.all);
    for (int k = 0; k < ORC_MAX_LEAVES; k++) free(pend[k].crumbs);
}

typedef struct {
    const uint64_t *st; int64_t n; int32_t num_itr; double cpuct, tau; int pre_expand, evaluator;
    const double *noise; int32_t noise_stride;
    uint32_t *visits; double *pi; int32_t *n_nodes; double *q;
    int tie_on; uint64_t tie_seed; int64_t tie_uid0;
    int leaves; int32_t *visited; int64_t *vl_left;
} leaves_job;

static void leaves_range(void *vj, int64_t lo, int64_t hi)
{
    leaves_job *jb = (leaves_job *)vj;
    for (int64_t i = lo; i < hi; i++) {
        uint64_t w[8];
        for (int k = 0; k < 8; k++) w[k] = jb->st[k * jb->n + i];
        uint64_t z = w[0] * 0x9E3779B97F4A7C15ull + w[1] * 0xC2B2AE3D27D4EB4Full + (w[4] & 0x0000FFFFFFFFFFFFull);   /* root hash */
        tie_rule tie = { jb->tie_on, jb->tie_seed, (uint64_t)(jb->tie_uid0 + i), (uint32_t)(z >> 32) ^ (uint32_t)z, 0 };
        mcts_search_leaves(w, jb->num_itr, jb->cpuct, jb->tau, jb->pre_expand, jb->leaves,
                           jb->noise ? jb->noise + i * jb->noise_stride : NULL, jb->evaluator == 0 ? eval_uniform : eval_hash,
                           jb->visits + i * ORC_NACT, jb->pi + i * ORC_NACT, jb->n_nodes ? jb->n_nodes + i : NULL,
                           jb->q ? jb->q + i * ORC_NACT : NULL, jb->tie_on ? &tie : NULL,
                           jb->visited ? jb->visited + i : NULL, jb->vl_left ? jb->vl_left + i : NULL);
    }
}

/* orc_mcts_batch / orc_mcts_batch_ties of the one-leaf oracle with `leaves` (1..16) selections per tree per round under
 * virtual loss; visited[n] (may be NULL): nodes reached by a selection, root included; vl_left[n] (may be NULL): virtual
 * losses left after the search */
void lvo_mcts_batch(const uint64_t *st, int64_t n, int32_t num_itr, double cpuct, double tau, int pre_expand,
                    int evaluator, const double *noise, int32_t noise_stride, uint32_t *visits, double *pi,
                    int32_t *n_nodes, double *q, int32_t nthreads, int tie_on, uint64_t tie_seed, int64_t tie_uid0,
                    int32_t leaves, int32_t *visited, int64_t *vl_left)
{
    leaves_job jb = { st, n, num_itr, cpuct, tau, pre_expand, evaluator, noise, noise_stride, visits, pi, n_nodes, q,
                      tie_on, tie_seed, tie_uid0, leaves, visited, vl_left };
    orc_parallel_for(leaves_range, &jb, n, nthreads);
}

/* the test evaluators on encoded positions: planes uint8[n][7][7][7] -> p[n][294], v[n] (0 = uniform, 1 = hash) */
void lvo_eval_batch(const uint8_t *planes, int64_t n, int evaluator, double *p, double *v)
{
    for (int64_t i = 0; i < n; i++)
        (evaluator == 0 ? eval_uniform : eval_hash)(NULL, (const uint8_t (*)[7][7])(planes + i * 343), p + i * ORC_NACT, v + i);
}
