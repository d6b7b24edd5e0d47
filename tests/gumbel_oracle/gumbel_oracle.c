/*
 * gumbel_oracle.c — CPU restatement of the engine's Gumbel search (include/ccx.h ccx_mcts_set_gumbel).  TEST
 * INFRASTRUCTURE, NOT PRODUCT: built by gumbel_oracle.py together with the one-leaf oracle's sources (oracle/ccx_oracle*.c,
 * for the board, encoding, Philox and thread-pool routines) into its own library.  It shares with the kernels only
 * csrc/ccx_fpmath.cuh (log, exp, the Gumbel draw) and csrc/ccx_gumbel_table.h (the sequential-halving schedule); the
 * Philox is the one-leaf oracle's, which the PUCT tests already hold equal to the kernels'.
 *
 * Same conventions as the leaves oracle: the reference's object formulation (eager child nodes), canonical edge order,
 * -ffp-contract=off, the two test evaluators.  Every expression below is the kernel's, evaluated left to right; every
 * float64 sum over a node's edges is warp_sum's order.
 */
#include "ccx_oracle.h"
#include "ccx_fpmath.cuh"
#include "ccx_gumbel_table.h"
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

uint64_t orc_planes_hash(const uint8_t planes[7][7][7]);        /* oracle/ccx_oracle_mcts.c */

#define GMAX 128

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

/* The kernels' float64 sum over a node's edges: lane l (0..31) sums x[l + 32c] for c = 0..3 in that order (0.0 past the
 * last edge), then an xor butterfly over offsets 16, 8, 4, 2, 1 adds lane l ^ off to lane l; every lane ends equal. */
static double warp_sum(const double *x, int ne)
{
    double s[32], t[32];
    for (int l = 0; l < 32; l++) {
        s[l] = 0.0;
        for (int c = 0; c < 4; c++) s[l] = s[l] + (l + 32 * c < ne ? x[l + 32 * c] : 0.0);
    }
    for (int off = 16; off; off >>= 1) {
        for (int l = 0; l < 32; l++) t[l] = s[l] + s[l ^ off];
        memcpy(s, t, sizeof(s));
    }
    return s[0];
}

typedef struct gnode gnode;
typedef struct {
    int in_player, idx;
    int64_t N;
    double W, Q, P;
    gnode *out;
} gedge;

struct gnode {
    orc_board state;
    int player, n_edges;
    double vraw;              /* evaluator value at the expansion */
    gedge *edges;
};

typedef struct { gnode **all; int n, cap; } garena;

typedef struct {
    int32_t m, S;
    double scale, c_visit, c_scale;
    uint64_t seed, uid;
    uint32_t serial;
    double g[GMAX];            /* root draws */
    int32_t mp;                /* m' */
    int32_t *table;            /* [m' rows][max(S, 1)] */
} gparams;

static gnode *gnew_node(garena *a, const orc_board *b, int player)
{
    gnode *nd = (gnode *)calloc(1, sizeof(gnode));
    nd->state = *b; nd->player = player;
    if (a->n == a->cap) { a->cap = a->cap ? a->cap * 2 : 1024; a->all = (gnode **)realloc(a->all, sizeof(gnode *) * (size_t)a->cap); }
    a->all[a->n++] = nd;
    return nd;
}

/* logits and sigma(q^) of a node's edges (the kernel's gumbel_node) */
typedef struct { double logit[GMAX], sigma[GMAX], maxlogit; int64_t nsum, nmax; } gstats;

static void node_stats(const gnode *nd, const gparams *gp, gstats *o)
{
    const int ne = nd->n_edges;
    double e[GMAX], a[GMAX], b[GMAX], q[GMAX];
    double mx = -INFINITY;
    o->nsum = 0; o->nmax = 0;
    for (int j = 0; j < ne; j++) {
        const gedge *ed = &nd->edges[j];
        o->logit[j] = fm_log(ed->P > DBL_MIN ? ed->P : DBL_MIN);
        mx = fmax(mx, o->logit[j]);
        o->nsum += ed->N;
        if (ed->N > o->nmax) o->nmax = ed->N;
    }
    o->maxlogit = mx;
    for (int j = 0; j < ne; j++) e[j] = fm_exp(o->logit[j] - mx);
    const double z = warp_sum(e, ne);
    for (int j = 0; j < ne; j++) {
        double pt = e[j] / z;
        pt = pt > DBL_MIN ? pt : DBL_MIN;
        a[j] = nd->edges[j].N > 0 ? pt : 0.0;
        b[j] = nd->edges[j].N > 0 ? pt * nd->edges[j].Q : 0.0;
    }
    const double sp = warp_sum(a, ne), spq = warp_sum(b, ne);
    const double ns = (double)o->nsum;
    const double vmix = o->nsum ? (nd->vraw + ns * spq / sp) / (1.0 + ns) : nd->vraw;
    double qmin = INFINITY, qmax = -INFINITY;
    for (int j = 0; j < ne; j++) {
        q[j] = nd->edges[j].N > 0 ? nd->edges[j].Q : vmix;
        qmin = fmin(qmin, q[j]);
        qmax = fmax(qmax, q[j]);
    }
    double den = qmax - qmin;
    den = den > 1e-8 ? den : 1e-8;
    const double vs = (gp->c_visit + (double)o->nmax) * gp->c_scale;
    for (int j = 0; j < ne; j++) o->sigma[j] = vs * ((q[j] - qmin) / den);
}

/* pi' = softmax(logit + sigma): w[j] / returned sum */
static double improved(const gnode *nd, const gstats *o, double *w)
{
    const int ne = nd->n_edges;
    double zz[GMAX], zmax = -INFINITY;
    for (int j = 0; j < ne; j++) { zz[j] = o->logit[j] + o->sigma[j]; zmax = fmax(zmax, zz[j]); }
    for (int j = 0; j < ne; j++) w[j] = fm_exp(zz[j] - zmax);
    return warp_sum(w, ne);
}

static double root_score(const gstats *o, int j, double g, int64_t N, int64_t cv)
{
    return N == cv ? fmax(-1e9, g + (o->logit[j] - o->maxlogit) + o->sigma[j]) : -INFINITY;
}

/* first maximal score; edge 0 when none is above -inf */
static int argmax_first(const double *s, int ne)
{
    double best = -INFINITY; int bi = -1;
    for (int j = 0; j < ne; j++) if (s[j] > best) { best = s[j]; bi = j; }
    return bi < 0 ? 0 : bi;
}

static int choose(const gnode *nd, int is_root, const gparams *gp)
{
    gstats o;
    double s[GMAX];
    node_stats(nd, gp, &o);
    const int ne = nd->n_edges;
    if (is_root) {
        const int cols = gp->S > 0 ? gp->S : 1;
        const int64_t k = o.nsum < cols - 1 ? o.nsum : cols - 1;
        const int64_t cv = gp->table[gp->mp * cols + k];
        for (int j = 0; j < ne; j++) s[j] = root_score(&o, j, gp->g[j], nd->edges[j].N, cv);
    } else {
        double w[GMAX];
        const double W = improved(nd, &o, w);
        const double d = 1.0 + (double)o.nsum;
        for (int j = 0; j < ne; j++) s[j] = w[j] / W - (double)nd->edges[j].N / d;
    }
    return argmax_first(s, ne);
}

static double gexpand(garena *a, gnode *leaf, orc_eval_fn eval)
{
    uint8_t planes[7][7][7];
    double p[ORC_NACT], v = 0.0;
    orc_to_model_input(&leaf->state, leaf->player, planes);
    eval(NULL, planes, p, &v);
    int8_t mv[6][ORC_MAX_DESTS][2]; int32_t cnt[6];
    orc_get_valid_moves(&leaf->state, leaf->player, mv, cnt);
    int total = 0;
    for (int id = 0; id < 6; id++) total += cnt[id];
    free(leaf->edges);
    leaf->n_edges = 0;
    leaf->edges = (gedge *)calloc((size_t)(total ? total : 1), sizeof(gedge));
    for (int id = 0; id < 6; id++) {
        qsort(mv[id], (size_t)cnt[id], 2, cmp_dest);
        int fr = leaf->state.pos[leaf->player - 1][id][0], fc = leaf->state.pos[leaf->player - 1][id][1];
        for (int k = 0; k < cnt[id]; k++) {
            gedge *e = &leaf->edges[leaf->n_edges++];
            int tr = mv[id][k][0], tc = mv[id][k][1];
            orc_board next = leaf->state;
            orc_place(&next, leaf->player, fr, fc, tr, tc);
            e->in_player = leaf->player;
            e->idx = id * 49 + tr * 7 + tc;
            e->P = p[e->idx];
            e->out = gnew_node(a, &next, 3 - leaf->player);
        }
    }
    leaf->vraw = v;
    return v;
}

static void gbackup(gedge **crumbs, int ncrumbs, const gnode *leaf, double v, int terminal)
{
    for (int i = 0; i < ncrumbs; i++) {
        gedge *e = crumbs[i];
        int same = e->in_player == leaf->player;
        e->N += 1;
        e->W += terminal ? 1.0 * (same ? -1 : 1) : v * (same ? 1 : -1);
        e->Q = e->W / (double)e->N;
    }
}

/* rounds = num_itr + pre_expand select / evaluate / expand / backup rounds (the first expands the root), S = rounds - 1 */
static void gumbel_search(const uint64_t rootw[8], int32_t rounds, gparams *gp, orc_eval_fn eval, uint32_t visits[ORC_NACT],
                          double pi[ORC_NACT], double q_out[ORC_NACT], int32_t *action, int32_t *n_nodes, int32_t *considered)
{
    garena a = {0};
    orc_board b; int tm;
    orc_unpack(rootw, &b, &tm, NULL);
    gnode *root = gnew_node(&a, &b, tm + 1);
    gedge **crumbs = (gedge **)malloc(sizeof(gedge *) * (size_t)(rounds + 2));
    memset(visits, 0, sizeof(uint32_t) * ORC_NACT);
    memset(pi, 0, sizeof(double) * ORC_NACT);
    memset(q_out, 0, sizeof(double) * ORC_NACT);
    for (int r = 0; r < rounds; r++) {
        gnode *cur = root;
        int nc = 0;
        while (cur->n_edges != 0) {
            gedge *e = &cur->edges[choose(cur, cur == root, gp)];
            crumbs[nc++] = e;
            cur = e->out;
        }
        if (orc_check_win(&cur->state)) { gbackup(crumbs, nc, cur, 0.0, 1); continue; }
        const double v = gexpand(&a, cur, eval);
        gbackup(crumbs, nc, cur, v, 0);
        if (cur == root) {
            for (int j = 0; j < root->n_edges; j++) {
                uint32_t out[4];
                orc_philox((uint32_t)gp->seed, (uint32_t)gp->uid, gp->serial, (uint32_t)j, (uint32_t)(gp->uid >> 32),
                           (uint32_t)(gp->seed >> 32), out);
                gp->g[j] = gp->scale * fm_gumbel(((uint64_t)out[1] << 32) | out[0]);
            }
            gp->mp = gp->m < root->n_edges ? gp->m : root->n_edges;
        }
    }
    *action = -1;
    if (considered) *considered = 0;
    for (int j = 0; j < root->n_edges; j++) {
        gedge *e = &root->edges[j];
        visits[e->idx] = (uint32_t)e->N;
        q_out[e->idx] = e->N ? e->W / (double)e->N : 0.0;
    }
    if (root->n_edges > 0) {
        gstats o;
        double w[GMAX], s[GMAX];
        node_stats(root, gp, &o);
        const double W = improved(root, &o, w);
        for (int j = 0; j < root->n_edges; j++) {
            pi[root->edges[j].idx] = w[j] / W;
            s[j] = root_score(&o, j, gp->g[j], root->edges[j].N, o.nmax);
        }
        *action = root->edges[argmax_first(s, root->n_edges)].idx;
        if (considered) {                                    /* bit mask of the m' top edges by g + logit, ties to the lower index */
            int taken[GMAX] = {0};
            for (int r = 0; r < gp->mp; r++) {
                int bi = -1;
                for (int j = 0; j < root->n_edges; j++)
                    if (!taken[j] && (bi < 0 || gp->g[j] + o.logit[j] > gp->g[bi] + o.logit[bi])) bi = j;
                taken[bi] = 1;
            }
            int32_t mask = 0;
            for (int j = 0; j < root->n_edges; j++) if (taken[j] && root->edges[j].idx == *action) mask = 1;
            *considered = mask;
        }
    }
    *n_nodes = a.n;
    for (int i = 0; i < a.n; i++) { free(a.all[i]->edges); free(a.all[i]); }
    free(a.all);
    free(crumbs);
}

typedef struct {
    const uint64_t *st; int64_t n; int32_t rounds, evaluator, m;
    double scale, c_visit, c_scale; uint64_t seed; int64_t uid0; const int64_t *uids;
    uint32_t *visits; double *pi, *q; int32_t *action, *n_nodes, *considered;
} gjob;

static void gumbel_range(void *vj, int64_t lo, int64_t hi)
{
    gjob *jb = (gjob *)vj;
    const int32_t S = jb->rounds > 0 ? jb->rounds - 1 : 0, cols = S > 0 ? S : 1;
    const int32_t rows = (jb->m < GMAX ? jb->m : GMAX) + 1;
    int32_t *table = (int32_t *)calloc((size_t)rows * cols, 4);
    for (int32_t r = 0; r < rows; r++) ccx_considered_visits(r, S, table + (size_t)r * cols);
    for (int64_t i = lo; i < hi; i++) {
        uint64_t w[8];
        for (int k = 0; k < 8; k++) w[k] = jb->st[k * jb->n + i];
        uint64_t z = w[0] * 0x9E3779B97F4A7C15ull + w[1] * 0xC2B2AE3D27D4EB4Full + (w[4] & 0x0000FFFFFFFFFFFFull);   /* root hash */
        gparams gp;
        memset(&gp, 0, sizeof(gp));
        gp.m = jb->m; gp.S = S; gp.scale = jb->scale; gp.c_visit = jb->c_visit; gp.c_scale = jb->c_scale; gp.seed = jb->seed;
        gp.uid = jb->uids ? (uint64_t)jb->uids[i] : (uint64_t)(jb->uid0 + i);
        gp.serial = (uint32_t)(z >> 32) ^ (uint32_t)z;
        gp.table = table;
        gumbel_search(w, jb->rounds, &gp, jb->evaluator == 0 ? eval_uniform : eval_hash, jb->visits + i * ORC_NACT,
                      jb->pi + i * ORC_NACT, jb->q + i * ORC_NACT, jb->action + i, jb->n_nodes + i,
                      jb->considered ? jb->considered + i : NULL);
    }
    free(table);
}

/* rounds = num_itr + pre_expand of BatchedMCTS; uids (may be NULL): tree uids, else uid0 + i; considered[n] (may be NULL):
 * 1 when the action is among the m' top root edges by g + logit */
void gmo_mcts_batch(const uint64_t *st, int64_t n, int32_t rounds, int32_t evaluator, int32_t m, double scale, double c_visit,
                    double c_scale, uint64_t seed, int64_t uid0, const int64_t *uids, uint32_t *visits, double *pi, double *q,
                    int32_t *action, int32_t *n_nodes, int32_t *considered, int32_t nthreads)
{
    gjob jb = { st, n, rounds, evaluator, m, scale, c_visit, c_scale, seed, uid0, uids, visits, pi, q, action, n_nodes, considered };
    orc_parallel_for(gumbel_range, &jb, n, nthreads);
}

void gmo_eval_batch(const uint8_t *planes, int64_t n, int evaluator, double *p, double *v)
{
    for (int64_t i = 0; i < n; i++)
        (evaluator == 0 ? eval_uniform : eval_hash)(NULL, (const uint8_t (*)[7][7])(planes + i * 343), p + i * ORC_NACT, v + i);
}

/* the shared header's functions, for the CPU tests */
double gmo_log(double x) { return fm_log(x); }
double gmo_exp(double x) { return fm_exp(x); }
void gmo_considered_visits(int32_t m, int32_t S, int32_t *out) { ccx_considered_visits(m, S, out); }
