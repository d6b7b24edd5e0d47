/*
 * reuse_oracle.c — CPU restatement of the engine's tree reuse (include/ccx.h ccx_mcts_begin_reuse) on top of the
 * leaf-parallel oracle.  TEST INFRASTRUCTURE, NOT PRODUCT: built by reuse_oracle.py into its own library together with the
 * one-leaf oracle's sources (oracle/ccx_oracle*.c).  The leaf-parallel oracle is included as source, so that its node and edge
 * types, descent, expansion, backup and test evaluators are the ones the persistent trees below use, and its lvo_* entry
 * points stay as they are.
 */
#include "../leaves_oracle/leaves_oracle.c"

/* ---- persistent trees (include/ccx.h ccx_mcts_begin_reuse) ----------------------------------------------------------------
 * A forest holds one tree per root across searches.  rvo_forest_begin restates the reuse begin: tree i starts from the
 * subtree of the node of its source tree (prev[i], default i) at depth 1 or 2 whose packed state words 0-4 equal the new root
 * (META's status byte masked), or fresh when the root is inactive, nothing matches, the match is unexpanded, the source was
 * inactive, the forest was invalidated (a new net) or would be reallocated (the engine's pool test), or the carry limit fails
 * (more than carry (S + 2) visited nodes, carry E edges or carry (S + 1) visits over the new root's edges).  A carried root
 * gets the root noise at once.  rvo_forest_search makes `sims` selections per active tree in rounds of up to `leaves` (one
 * while the root is unexpanded; the root's expansion mixes in the noise), as mcts_search_leaves does; the tie rule's
 * simulation index counts the selections of the current search. */
typedef struct {
    varena a;
    vnode *root;              /* NULL: inactive */
    uint32_t serial, sim;
} vtree;

typedef struct {
    int64_t n, cap;
    int32_t npt, ept, pm;     /* pool budgets of the engine's trees_reserve: a begin that needs more starts every tree fresh */
    int valid;                /* 0 after rvo_forest_invalidate and before the first begin */
    vtree *t;
} rvo_forest;

static void vtree_free(vtree *t)
{
    for (int i = 0; i < t->a.n; i++) { free(t->a.all[i]->edges); free(t->a.all[i]); }
    free(t->a.all);
    memset(t, 0, sizeof(*t));
}

rvo_forest *rvo_forest_new(void) { return (rvo_forest *)calloc(1, sizeof(rvo_forest)); }

void rvo_forest_free(rvo_forest *f)
{
    for (int64_t i = 0; i < f->n; i++) vtree_free(&f->t[i]);
    free(f->t);
    free(f);
}

void rvo_forest_invalidate(rvo_forest *f) { f->valid = 0; }

static vnode *vcopy(varena *a, const vnode *s)
{
    vnode *d = vnew_node(a, &s->state, s->player);
    d->visited = s->visited;
    d->n_edges = s->n_edges;
    if (s->edges) {
        d->edges = (vedge *)calloc((size_t)(s->n_edges ? s->n_edges : 1), sizeof(vedge));
        for (int i = 0; i < s->n_edges; i++) {
            d->edges[i] = s->edges[i];
            d->edges[i].out = vcopy(a, s->edges[i].out);
        }
    }
    return d;
}

static void vcount(const vnode *nd, int64_t *visited, int64_t *edges)
{
    *visited += nd->visited;
    *edges += nd->n_edges;
    for (int i = 0; i < nd->n_edges; i++) vcount(nd->edges[i].out, visited, edges);
}

static int vsame(const vnode *nd, const uint64_t w[5])
{
    uint64_t x[8];
    orc_pack(&nd->state, nd->player - 1, 0, x);
    return x[0] == w[0] && x[1] == w[1] && x[2] == w[2] && x[3] == w[3] && (x[4] & 0x00FFFFFFFFFFFFFFull) == w[4];
}

/* the engine's mix_root_noise: lane-strided partial sums, then a butterfly over the 32 lanes */
static void vmix_noise(vnode *root, const double *noise, int normalize)
{
    double scale = 1.0;
    if (normalize) {
        double s[32];
        for (int l = 0; l < 32; l++) { s[l] = 0.0; for (int j = l; j < root->n_edges; j += 32) s[l] += noise[j]; }
        for (int off = 16; off; off >>= 1) {
            double t[32];
            for (int l = 0; l < 32; l++) t[l] = s[l] + s[l ^ off];
            memcpy(s, t, sizeof(s));
        }
        scale = s[0] > 0.0 ? 1.0 / s[0] : 0.0;
    }
    for (int j = 0; j < root->n_edges; j++) {
        double nz = normalize ? noise[j] * scale : noise[j];
        root->edges[j].P = root->edges[j].P * (1. - 0.25) + 0.25 * nz;
    }
}

static uint32_t root_hash(const uint64_t w[8])
{
    uint64_t z = w[0] * 0x9E3779B97F4A7C15ull + w[1] * 0xC2B2AE3D27D4EB4Full + (w[4] & 0x0000FFFFFFFFFFFFull);
    return (uint32_t)(z >> 32) ^ (uint32_t)z;
}

/* reused[n] (may be NULL) as the engine reports it: 1 / 2 = depth of the match, 0 = fresh, -2 = inactive */
void rvo_forest_begin(rvo_forest *f, const uint64_t *st, int64_t n, int32_t S, int32_t edges_per_tree, int32_t min_ply,
                      int32_t ply_parity, int32_t carry, const int64_t *prev, const double *noise, int32_t noise_stride,
                      int32_t noise_normalize, int32_t *reused)
{
    const int64_t E = edges_per_tree > 0 ? edges_per_tree : 64 * ((int64_t)S + 1);
    const int32_t npt = (1 + carry) * (S + 2), ept = (int32_t)((1 + carry) * E), pm = (1 + carry) * (S + 2);
    int keep = f->valid && f->cap >= n && f->npt >= npt && f->ept == ept && f->pm >= pm;
    if (!keep) { f->cap = n; f->npt = npt; f->ept = ept; f->pm = pm; }
    vtree *nt = (vtree *)calloc((size_t)(n ? n : 1), sizeof(vtree));
    for (int64_t i = 0; i < n; i++) {
        uint64_t w[8];
        for (int k = 0; k < 8; k++) w[k] = st[k * n + i];
        const uint64_t m = w[4];
        int inactive = min_ply >= 0 && ((m >> 56) != 0 || (int)((m >> 32) & 0xFFFF) < min_ply);
        if (ply_parity >= 0 && (int)((m >> 32) & 1) != ply_parity) inactive = 1;
        vtree *t = &nt[i];
        t->serial = root_hash(w);
        int kind = inactive ? -2 : 0;
        const int64_t s = prev ? prev[i] : i;
        if (!inactive && keep && s >= 0 && s < f->n && f->t[s].root) {
            const vnode *sr = f->t[s].root;
            uint64_t key[5] = { w[0], w[1], w[2], w[3], w[4] & 0x00FFFFFFFFFFFFFFull };
            const vnode *hit = NULL;
            int depth = 0;
            for (int a = 0; a < sr->n_edges && !hit; a++) {
                const vnode *c = sr->edges[a].out;
                if (vsame(c, key)) { hit = c; depth = 1; }
                for (int b = 0; b < c->n_edges && !hit; b++)
                    if (vsame(c->edges[b].out, key)) { hit = c->edges[b].out; depth = 2; }
            }
            if (hit && hit->n_edges > 0) {
                int64_t nsum = 0, nodes = 0, edges = 0;
                for (int j = 0; j < hit->n_edges; j++) nsum += hit->edges[j].N;
                vcount(hit, &nodes, &edges);
                if (nsum <= (int64_t)carry * (S + 1) && nodes <= (int64_t)carry * (S + 2) && edges <= (int64_t)carry * E) {
                    t->root = vcopy(&t->a, hit);
                    if (noise) vmix_noise(t->root, noise + i * noise_stride, noise_normalize);
                    kind = depth;
                }
            }
        }
        if (!inactive && !t->root) {
            orc_board b; int tm;
            orc_unpack(w, &b, &tm, NULL);
            t->root = vnew_node(&t->a, &b, tm + 1);
            t->root->visited = 1;
        }
        if (reused) reused[i] = kind;
    }
    for (int64_t i = 0; i < f->n; i++) vtree_free(&f->t[i]);
    free(f->t);
    f->t = nt; f->n = n; f->valid = 1;
}

typedef struct {
    rvo_forest *f; int32_t sims, leaves; double cpuct; int evaluator;
    const double *noise; int32_t noise_stride, noise_normalize; int tie_on; uint64_t tie_seed; int64_t tie_uid0;
} forest_job;

static void forest_search_range(void *vj, int64_t lo, int64_t hi)
{
    forest_job *jb = (forest_job *)vj;
    orc_eval_fn eval = jb->evaluator == 0 ? eval_uniform : eval_hash;
    for (int64_t i = lo; i < hi; i++) {
        vtree *t = &jb->f->t[i];
        if (!t->root) continue;
        vnode *root = t->root;
        tie_rule tie = { jb->tie_on, jb->tie_seed, (uint64_t)(jb->tie_uid0 + i), t->serial, 0 };
        struct { vnode *leaf; vedge **crumbs; int ncrumbs, dup_of; double v; } pend[ORC_MAX_LEAVES];
        const int pmax = jb->f->pm + 2;
        for (int k = 0; k < ORC_MAX_LEAVES; k++) pend[k].crumbs = (vedge **)malloc(sizeof(vedge *) * (size_t)pmax);
        int done = 0;
        while (done < jb->sims) {
            int m = root->n_edges == 0 ? 1 : (jb->sims - done < jb->leaves ? jb->sims - done : jb->leaves);
            int np = 0;
            for (int k = 0; k < m; k++) {
                tie.sim = t->sim++;
                done++;
                int nc;
                vnode *leaf = vmove_to_leaf(root, jb->cpuct, pend[np].crumbs, &nc, &tie);
                leaf->visited = 1;
                if (orc_check_win(&leaf->state)) { vbackup(pend[np].crumbs, nc, leaf, 0.0, 1, 0); continue; }
                int dup = -1;
                for (int j = 0; j < np && dup < 0; j++) if (pend[j].leaf == leaf) dup = j;
                pend[np].leaf = leaf; pend[np].ncrumbs = nc; pend[np].dup_of = dup;
                for (int c = 0; c < nc; c++) pend[np].crumbs[c]->V += 1;
                np++;
            }
            for (int j = 0; j < np; j++) {
                if (pend[j].dup_of < 0) pend[j].v = vexpand(&t->a, pend[j].leaf, eval, NULL);
                else pend[j].v = pend[pend[j].dup_of].v;
                vbackup(pend[j].crumbs, pend[j].ncrumbs, pend[j].leaf, pend[j].v, 0, 1);
            }
            if (jb->noise && np > 0 && pend[0].leaf == root && pend[0].dup_of < 0)
                vmix_noise(root, jb->noise + i * jb->noise_stride, jb->noise_normalize);
        }
        for (int k = 0; k < ORC_MAX_LEAVES; k++) free(pend[k].crumbs);
    }
}

void rvo_forest_search(rvo_forest *f, int32_t sims, int32_t leaves, double cpuct, int evaluator, const double *noise,
                       int32_t noise_stride, int32_t noise_normalize, int tie_on, uint64_t tie_seed, int64_t tie_uid0, int32_t nthreads)
{
    forest_job jb = { f, sims, leaves, cpuct, evaluator, noise, noise_stride, noise_normalize, tie_on, tie_seed, tie_uid0 };
    orc_parallel_for(forest_search_range, &jb, f->n, nthreads);
}

/* ccx_mcts_finalize of every tree (node count = edges + 1, -2 for an inactive tree); vl_left (may be NULL): virtual losses left;
 * N, W, P (may be NULL): [n][ORC_NACT] root edge statistics by policy index */
void rvo_forest_finalize(const rvo_forest *f, double tau, uint32_t *visits, double *pi, double *q, int32_t *n_nodes, int64_t *vl_left,
                         double *W, double *P)
{
    for (int64_t i = 0; i < f->n; i++) {
        uint32_t *vi = visits + i * ORC_NACT; double *pii = pi + i * ORC_NACT, *qi = q + i * ORC_NACT;
        memset(vi, 0, sizeof(uint32_t) * ORC_NACT); memset(pii, 0, sizeof(double) * ORC_NACT); memset(qi, 0, sizeof(double) * ORC_NACT);
        if (W) memset(W + i * ORC_NACT, 0, sizeof(double) * ORC_NACT);
        if (P) memset(P + i * ORC_NACT, 0, sizeof(double) * ORC_NACT);
        const vnode *root = f->t[i].root;
        if (vl_left) vl_left[i] = 0;
        if (!root) { n_nodes[i] = -2; continue; }
        double sum = 0.0;
        for (int j = 0; j < root->n_edges; j++) {
            const vedge *e = &root->edges[j];
            vi[e->idx] = (uint32_t)e->N;
            pii[e->idx] = pow((double)e->N, 1. / tau);
            qi[e->idx] = e->Q;
            if (W) W[i * ORC_NACT + e->idx] = e->W;
            if (P) P[i * ORC_NACT + e->idx] = e->P;
        }
        for (int a = 0; a < ORC_NACT; a++) sum += pii[a];
        if (sum > 0) for (int a = 0; a < ORC_NACT; a++) pii[a] /= sum;
        int64_t nodes = 0, edges = 0;
        vcount(root, &nodes, &edges);
        n_nodes[i] = (int32_t)(edges + 1);
        if (vl_left)
            for (int k = 0; k < f->t[i].a.n; k++)
                for (int j = 0; j < f->t[i].a.all[k]->n_edges; j++) vl_left[i] += f->t[i].a.all[k]->edges[j].V;
    }
}

/* root edge statistics of the child reached by policy index `act` from tree i's root: N, W, P [ORC_NACT] by the child's
 * policy indices (zero when the child is unexpanded) — what a carried tree's root must hold */
void rvo_forest_child_stats(const rvo_forest *f, int64_t i, int32_t act, uint32_t *N, double *W, double *P)
{
    memset(N, 0, sizeof(uint32_t) * ORC_NACT); memset(W, 0, sizeof(double) * ORC_NACT); memset(P, 0, sizeof(double) * ORC_NACT);
    const vnode *root = f->t[i].root;
    if (!root) return;
    for (int j = 0; j < root->n_edges; j++) {
        if (root->edges[j].idx != act) continue;
        const vnode *c = root->edges[j].out;
        for (int k = 0; k < c->n_edges; k++) {
            N[c->edges[k].idx] = (uint32_t)c->edges[k].N; W[c->edges[k].idx] = c->edges[k].W; P[c->edges[k].idx] = c->edges[k].P;
        }
    }
}
