/* TEST INFRASTRUCTURE — see pastar_oracle.h.  Plain C, scalar, one thread.
 * Build: gcc -std=c11 -O2 -ffp-contract=off (the weight routine is float-order
 * sensitive; the reference is built without FMA: Makefile:53 has -O3 only). */
#include "pastar_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------ */
/* Cost model — Cost.cpp:12-271, Cost.h:13,49                               */
/* The reference fills pam250[a][b] with 17 - (Dayhoff PAM250 score) for    */
/* the 20 amino acids and 12 for DASH against 17 of them (not C, S, T);     */
/* everything else stays 0.  The scores below are the published PAM250      */
/* matrix (lower triangle) in the order the reference lists the residues.   */
/* ------------------------------------------------------------------------ */
static const char PO_AA[21] = "CSTPAGNDEQHRKMILVFYW";
static const signed char PO_PAM250[20][20] = {
    /*C*/ {12},
    /*S*/ {0, 2},
    /*T*/ {-2, 1, 3},
    /*P*/ {-3, 1, 0, 6},
    /*A*/ {-2, 1, 1, 1, 2},
    /*G*/ {-3, 1, 0, -1, 1, 5},
    /*N*/ {-4, 1, 0, -1, 0, 0, 2},
    /*D*/ {-5, 0, 0, -1, 0, 1, 2, 4},
    /*E*/ {-5, 0, 0, -1, 0, 0, 1, 3, 4},
    /*Q*/ {-5, -1, -1, 0, 0, -1, 1, 2, 2, 4},
    /*H*/ {-3, -1, -1, 0, -1, -2, 2, 1, 1, 3, 6},
    /*R*/ {-4, 0, -1, 0, -2, -3, 0, -1, -1, 1, 2, 6},
    /*K*/ {-5, 0, 0, -1, -1, -2, 1, 0, 0, 1, 0, 3, 5},
    /*M*/ {-5, -2, -1, -2, -1, -3, -2, -3, -2, -1, -2, 0, 0, 6},
    /*I*/ {-2, -1, 0, -2, -1, -3, -2, -2, -2, -2, -2, -2, -2, 2, 5},
    /*L*/ {-6, -3, -2, -3, -2, -4, -3, -4, -3, -2, -2, -3, -3, 4, 2, 6},
    /*V*/ {-2, -1, 0, -1, 0, -1, -2, -2, -2, -2, -2, -2, -2, 2, 4, 2, 4},
    /*F*/ {-4, -3, -3, -5, -4, -5, -4, -6, -5, -5, -2, -4, -5, 0, 1, 2, -1, 9},
    /*Y*/ {0, -3, -3, -5, -3, -5, -2, -4, -4, -4, 0, -4, -4, -2, -1, -1, -2, 7, 10},
    /*W*/ {-8, -2, -5, -6, -6, -7, -4, -7, -7, -5, -3, 2, -3, -4, -5, -2, -6, 0, 0, 17},
};

static int32_t g_cost[90 * 90];
static int g_cost_ready = 0;

static void cost_init(void)
{
    if (g_cost_ready) return;
    memset(g_cost, 0, sizeof(g_cost));
    for (int i = 0; i < 20; i++)
        for (int j = 0; j <= i; j++) {
            int a = PO_AA[i], b = PO_AA[j];
            g_cost[a * 90 + b] = g_cost[b * 90 + a] = 17 - PO_PAM250[i][j];
        }
    /* Cost.cpp:15-31: DASH rows, 17 residues */
    for (const char *c = "PAGNDEQHRKMILVFYW"; *c; c++) g_cost['-' * 90 + *c] = g_cost[*c * 90 + '-'] = 12;
    g_cost_ready = 1;
}

void po_cost_table(int32_t out[90 * 90])
{
    cost_init();
    memcpy(out, g_cost, sizeof(g_cost));
}

int po_cost(int a, int b) /* Cost.cpp:267-271 */
{
    cost_init();
    return g_cost[a * 90 + b];
}

/* ------------------------------------------------------------------------ */
/* Pairwise reverse DP — PairAlign.cpp:96-171                               */
/* ------------------------------------------------------------------------ */
enum { NoGap, GapX, GapY }; /* PairAlign.h:24 */

void po_pair_table(const char *s1, int l1, const char *s2, int l2, int32_t *m)
{
    cost_init();
    int cols = l2 + 1;
    int *aff = (int *)malloc(sizeof(int) * (size_t)(l1 + 1) * cols);
#define M(i, j) m[(size_t)(i) * cols + (j)]
#define A(i, j) aff[(size_t)(i) * cols + (j)]
    /* borders, PairAlign.cpp:142-160 (guards added for empty strings, which
       the reference would index out of range) */
    M(l1, l2) = 0;
    A(l1, l2) = NoGap;
    if (l2 >= 1) {
        M(l1, l2 - 1) = PO_GAP_OPEN;
        A(l1, l2 - 1) = GapY;
    }
    if (l1 >= 1) {
        M(l1 - 1, l2) = PO_GAP_OPEN;
        A(l1 - 1, l2) = GapX;
    }
    for (int j = l2 - 2; j >= 0; j--) {
        M(l1, j) = M(l1, j + 1) + PO_GAP_EXTENSION;
        A(l1, j) = GapY;
    }
    for (int i = l1 - 2; i >= 0; i--) {
        M(i, l2) = M(i + 1, l2) + PO_GAP_EXTENSION;
        A(i, l2) = GapX;
    }
    /* interior, PairAlign.cpp:107-134,162-168 */
    for (int i = l1 - 1; i >= 0; i--) {
        for (int j = l2 - 1; j >= 0; j--) {
            int min_value, gap_value;
            int c0 = M(i + 1, j) + (A(i + 1, j) == GapX ? PO_GAP_EXTENSION : PO_GAP_OPEN);
            int c1 = M(i, j + 1) + (A(i, j + 1) == GapY ? PO_GAP_EXTENSION : PO_GAP_OPEN);
            if (c0 < c1) {
                min_value = c0;
                gap_value = GapX;
            } else {
                min_value = c1;
                gap_value = GapY;
            }
            int c2 = M(i + 1, j + 1) + g_cost[(unsigned char)s1[i] * 90 + (unsigned char)s2[j]];
            if (c2 < min_value) {
                min_value = c2;
                gap_value = NoGap;
            }
            M(i, j) = min_value;
            A(i, j) = gap_value;
        }
    }
#undef M
#undef A
    free(aff);
}

/* ------------------------------------------------------------------------ */
/* Altschul rationale-2 pair weights — WeightedSP.cpp                        */
/* ------------------------------------------------------------------------ */
#define W_BIG 999999     /* WeightedSP.hpp:13 */
#define W_GAPCOST 8      /* :18 */
#define W_EFF_GAPCOST 0  /* :22 */
enum { W_DIAG = 0, W_VERT = 1, W_HORZ = 2 };

typedef struct tnode {
    struct tnode *parent, *left, *right, *brother;
    float weight, w, W, v, V;
    int seq; /* >=0 leaf, -1 internal, -2 root */
} tnode;

static int min_of3(int a, int b, int c) /* WeightedSP.cpp:21-35 */
{
    if (a < b) return a < c ? a : c;
    return b < c ? b : c;
}

/* WeightedSP.cpp:109-142.  s1/s2 are the dash-prefixed strings. */
static float path_to_cost(const char *s1, const char *s2, int n, int m, int **dd, int **hh, int **vv)
{
    int i, j, V, H, Mv;
    int dir = W_DIAG, match = 0;
    for (i = n, j = m; (i || j);) {
        V = vv[i][j] - (dir == W_VERT ? (j == m ? W_EFF_GAPCOST : W_GAPCOST) : 0);
        H = hh[i][j] - (dir == W_HORZ ? (i == n ? W_EFF_GAPCOST : W_GAPCOST) : 0);
        Mv = min_of3(V, H, dd[i][j]);
        if (!j || Mv == V) {
            dir = W_VERT;
            --i;
        } else if (!i || Mv == H) {
            dir = W_HORZ;
            --j;
        } else {
            dir = W_DIAG;
            match += s1[i] == s2[j];
            --i;
            --j;
        }
    }
    int ret = ((int)(0.5 + 1000.0 * (n - match + m - match) / (n + m)));
    return (float)ret;
}

static int **alloc2(int r, int c)
{
    int **p = (int **)malloc(sizeof(int *) * r);
    for (int i = 0; i < r; i++) p[i] = (int *)calloc((size_t)c, sizeof(int));
    return p;
}
static void free2(int **p, int r)
{
    for (int i = 0; i < r; i++) free(p[i]);
    free(p);
}

/* WeightedSP.cpp:144-244.  seqs[] are dash-prefixed, NUL-terminated; Dij n x n. */
static void primer(int num, char **seqs, const int *plen, float *Dij)
{
    int maxl = 0;
    for (int i = 0; i < num; i++)
        if (plen[i] > maxl) maxl = plen[i];
    int **dd = alloc2(maxl + 2, maxl + 2), **hh = alloc2(maxl + 2, maxl + 2), **vv = alloc2(maxl + 2, maxl + 2);
    for (int I = 0; I < num - 1; I++) {
        const char *sa = seqs[I];
        int n = plen[I];
        for (int J = I + 1; J < num; J++) {
            const char *sb = seqs[J];
            int m = plen[J];
            int i, j, Gi, Gj;
            dd[0][0] = 0;
            hh[0][0] = vv[0][0] = W_EFF_GAPCOST;
            for (j = 1; j <= m; j++) { /* j == m reads the string terminator: cost 0 */
                vv[0][j] = dd[0][j] = W_BIG;
                hh[0][j] = hh[0][j - 1] + po_cost('-', (unsigned char)sb[j]);
            }
            for (i = 1; i <= n; i++) {
                hh[i][0] = dd[i][0] = W_BIG;
                vv[i][0] = vv[i - 1][0] + po_cost((unsigned char)sa[i], '-');
            }
            for (i = 1; i < n; i++) {
                Gi = (i == (n - 1) ? W_EFF_GAPCOST : W_GAPCOST);
                for (j = 1; j < m; j++) {
                    Gj = (j == (m - 1) ? W_EFF_GAPCOST : W_GAPCOST);
                    dd[i][j] = min_of3(dd[i - 1][j - 1], hh[i - 1][j - 1], vv[i - 1][j - 1]) +
                               po_cost((unsigned char)sa[i], (unsigned char)sb[j]);
                    hh[i][j] = min_of3(dd[i][j - 1] + Gi, hh[i][j - 1], vv[i][j - 1] + Gi) +
                               po_cost('-', (unsigned char)sb[j]);
                    vv[i][j] = min_of3(dd[i - 1][j] + Gj, hh[i - 1][j] + Gj, vv[i - 1][j]) +
                               po_cost((unsigned char)sa[i], '-');
                }
            }
            float d = path_to_cost(sa, sb, n - 1, m - 1, dd, hh, vv);
            if (d <= 0) d = 1; /* :227-228 */
            Dij[J * num + I] = Dij[I * num + J] = d;
        }
    }
    free2(dd, maxl + 2);
    free2(hh, maxl + 2);
    free2(vv, maxl + 2);
}

typedef struct {
    tnode **tree;
    int tree_n;
    const float *Dij;
    int num;
} njctx;

/* WeightedSP.cpp:248-266 */
static float path_cost_rec(const njctx *c, const tnode *A, const tnode *B, int *path_length)
{
    if (A->seq < 0) {
        ++(*path_length);
        float a = path_cost_rec(c, A->left, B, path_length);
        float b = path_cost_rec(c, A->right, B, path_length);
        return a + b;
    } else if (B->seq < 0) {
        ++(*path_length);
        float a = path_cost_rec(c, A, B->left, path_length);
        float b = path_cost_rec(c, A, B->right, path_length);
        return a + b;
    }
    return c->Dij[A->seq * c->num + B->seq];
}
/* WeightedSP.cpp:270-277, 281-288 */
static float path_cost_n(const njctx *c, const tnode *A, const tnode *B)
{
    int path_length = 1;
    float cost = path_cost_rec(c, A, B, &path_length);
    return (float)(cost / path_length);
}
static float path_cost(const njctx *c, int i, int j) { return path_cost_n(c, c->tree[i], c->tree[j]); }

/* WeightedSP.cpp:57-63 */
static float cost_to_leafs(const tnode *A, float total, int *count2)
{
    if (A->seq >= 0) return (total + A->weight);
    (*count2)++;
    float a = cost_to_leafs(A->left, A->weight + total, count2);
    float b = cost_to_leafs(A->right, A->weight + total, count2);
    return a + b;
}

/* WeightedSP.cpp:65-78.  `f(&count2)/count2`: g++ evaluates the call first,
 * so the divisor is the post-call count (checked against oracle/_ref). */
static float curr_cost(const njctx *c, int i, int j)
{
    float diz = 0.0f, djz = 0.0f;
    int count2 = 1, rem = c->tree_n;
    for (int t = 0; t < rem; ++t)
        if (t != i && t != j) {
            diz += path_cost(c, i, t);
            djz += path_cost(c, j, t);
        }
    diz = diz / (rem - 2);
    djz = djz / (rem - 2);
    float pc = path_cost(c, i, j);
    float ctl = cost_to_leafs(c->tree[i], 0.0f, &count2);
    return ((pc + diz - djz) / 2 - ctl / count2);
}

/* WeightedSP.cpp:290-311 */
static float compute_S(const njctx *c, int i, int j, int numNodes)
{
    float s1 = 0, s2 = 0;
    for (int t = 0; t < numNodes; t++)
        if (t != i && t != j) {
            float a = path_cost(c, i, t);
            float b = path_cost(c, j, t);
            s1 += a + b;
        }
    s1 = s1 / (2 * (numNodes - 2));
    for (int t = 0; t < numNodes - 1; t++)
        for (int tt = t + 1; tt < numNodes; tt++)
            if (t != i && t != j && tt != i && tt != j) s2 += path_cost(c, t, tt);
    s2 = s2 / (numNodes - 2);
    float total = (s1 + s2 + path_cost(c, i, j) / 2);
    return total;
}

static tnode *new_node(tnode *left, tnode *right, int seq) /* WeightedSP.hpp:31-52 with the args the callers pass */
{
    tnode *t = (tnode *)calloc(1, sizeof(tnode));
    t->left = left;
    t->right = right;
    t->weight = 0.0f;
    t->seq = seq;
    return t;
}

/* WeightedSP.cpp:403-420 */
static void weights_from_tree(float product, float sum, const tnode *no, const tnode *brother, float *wm, int num,
                              int from_seq)
{
    if (no->seq > -1) {
        wm[from_seq * num + no->seq] = sum * product;
    } else if (brother == NULL) {
        weights_from_tree(product * no->left->W, sum + no->right->weight, no->right, NULL, wm, num, from_seq);
        weights_from_tree(product * no->right->W, sum + no->left->weight, no->left, NULL, wm, num, from_seq);
    } else {
        weights_from_tree(product * no->V, sum + brother->weight, brother, NULL, wm, num, from_seq);
        if (no->seq != -2) weights_from_tree(product * brother->W, sum + no->weight, no->parent, no->brother, wm, num, from_seq);
    }
}

int po_weights(int num, const char *const *seqs_in, const int *lens, float *out)
{
    cost_init();
    for (int i = 0; i < num; i++)
        if (lens[i] > 998) return -1; /* F4: WeightedSP.cpp:148 fixed 1000x1000 scratch */
    /* :447 — prefix every sequence with a dash */
    char **seqs = (char **)malloc(sizeof(char *) * num);
    int *plen = (int *)malloc(sizeof(int) * num);
    for (int i = 0; i < num; i++) {
        plen[i] = lens[i] + 1;
        seqs[i] = (char *)malloc((size_t)plen[i] + 1);
        seqs[i][0] = '-';
        memcpy(seqs[i] + 1, seqs_in[i], (size_t)lens[i]);
        seqs[i][plen[i]] = 0;
    }
    float *Dij = (float *)calloc((size_t)num * num, sizeof(float));
    float *wm = (float *)calloc((size_t)num * num, sizeof(float));
    primer(num, seqs, plen, Dij);

    /* phylogeneticThreeNeighborJoin, :317-401 */
    int cap = 2 * num + 2;
    tnode **tree = (tnode **)malloc(sizeof(tnode *) * cap);
    tnode **list = (tnode **)malloc(sizeof(tnode *) * cap);
    int tree_n = 0, list_n = 0;
    for (int i = 0; i < num; i++) {
        tnode *t = new_node(NULL, NULL, i);
        tree[tree_n++] = t;
        list[list_n++] = t;
    }
    njctx c = {tree, tree_n, Dij, num};
    int rem = num;
    float minv = (float)1.0E20;
    int min_i = 0, min_j = 0;
    while (rem > 2) {
        for (int i = 0; i < rem - 1; i++)
            for (int j = i + 1; j < rem; j++) {
                float tmp = compute_S(&c, i, j, rem);
                if (tmp < minv) {
                    min_i = i;
                    min_j = j;
                    minv = tmp;
                }
            }
        /* join_nodes, :80-107 */
        tnode *l = tree[min_i];
        l->weight = curr_cost(&c, min_i, min_j);
        tnode *r = tree[min_j];
        r->weight = curr_cost(&c, min_j, min_i);
        tnode *nn = new_node(l, r, -1);
        l->brother = r;
        r->brother = l;
        l->parent = r->parent = nn;
        list[list_n++] = nn;
        tree[min_i] = nn;
        tree[min_j] = tree[c.tree_n - 1];
        c.tree_n--;
        rem--;
        minv = (float)1.0E20;
    }
    tnode *l = tree[0], *r = tree[1];
    tnode *anc = new_node(l, r, -2);
    l->brother = r;
    r->brother = l;
    l->parent = r->parent = anc;
    list[list_n++] = anc;
    {
        int count2 = 1;
        float len = path_cost_n(&c, l, r);
        float a = cost_to_leafs(l, 0.0f, &count2);
        len -= a / count2;
        count2 = 1;
        float b = cost_to_leafs(r, 0.0f, &count2);
        len -= b / count2;
        anc->left->weight = len;
    }

    /* weightAltschulsRationale2, :464-496 */
    int p = 0;
    tnode *no = NULL;
    for (; list[p]->seq > -1; ++p) {
        no = list[p];
        no->w = 1.0f;
        no->W = no->weight;
    }
    for (; (no = list[p])->seq > -2; ++p) {
        no->w = no->left->w * no->right->W + no->left->W * no->right->w;
        no->W = no->weight * no->w + no->left->W * no->right->W;
    }
    no->V = 1;
    no->v = 0;
    do {
        no = list[--p];
        no->v = no->parent->v * no->brother->W + no->parent->V * no->brother->w;
        no->V = no->weight * no->v + no->parent->V * no->brother->W;
    } while (p != 0);
    for (; (no = list[p])->seq > -1; ++p) weights_from_tree(1.0f, no->weight, no->parent, no->brother, wm, num, no->seq);

    /* :498-509 — scale so the smallest is about 8 */
    float sm = 1.0E+30f;
    for (int j = 1; j < num; ++j)
        for (int i = 0; i < j; ++i)
            if (wm[i * num + j] < sm) sm = wm[i * num + j];
    sm = (float)((double)sm / 7.9);
    for (int i = 0; i < num * num; i++) out[i] = 0.0f;
    for (int i = 0; i < num - 1; ++i)
        for (int j = i + 1; j < num; ++j) out[i * num + j] = out[j * num + i] = (float)((double)(wm[i * num + j] / sm) + 0.5);

    for (int i = 0; i < list_n; i++) free(list[i]);
    free(list);
    free(tree);
    free(Dij);
    free(wm);
    for (int i = 0; i < num; i++) free(seqs[i]);
    free(seqs);
    free(plen);
    return 0;
}

/* ------------------------------------------------------------------------ */
/* Problem                                                                   */
/* ------------------------------------------------------------------------ */
struct po_problem {
    int n, npairs;
    int len[PO_MAX_SEQ];
    char *seq[PO_MAX_SEQ]; /* NUL terminated: getNeigh reads seq[len] (F14) */
    int32_t *table[PO_MAX_SEQ * PO_MAX_SEQ];
    int pa[PO_MAX_SEQ * PO_MAX_SEQ], pb[PO_MAX_SEQ * PO_MAX_SEQ];
    int32_t w[PO_MAX_SEQ * PO_MAX_SEQ]; /* (int)weightMatrix[i][j] */
};

po_problem *po_create(int n, const char *const *seqs, const int *lens, const int32_t *w_int)
{
    if (n < 2 || n > PO_MAX_SEQ) return NULL;
    po_problem *p = (po_problem *)calloc(1, sizeof(po_problem));
    p->n = n;
    for (int i = 0; i < n; i++) {
        p->len[i] = lens[i];
        p->seq[i] = (char *)calloc((size_t)lens[i] + 1, 1);
        memcpy(p->seq[i], seqs[i], (size_t)lens[i]);
    }
    /* HeuristicHPair.cpp:54-61: pairs in (i<j) order */
    for (int i = 0; i < n - 1; i++)
        for (int j = i + 1; j < n; j++) {
            int k = p->npairs++;
            p->pa[k] = i;
            p->pb[k] = j;
            p->table[k] = (int32_t *)malloc(sizeof(int32_t) * (size_t)(lens[i] + 1) * (size_t)(lens[j] + 1));
            po_pair_table(p->seq[i], lens[i], p->seq[j], lens[j], p->table[k]);
        }
    if (w_int) {
        memcpy(p->w, w_int, sizeof(int32_t) * (size_t)n * n);
    } else {
        float *wf = (float *)malloc(sizeof(float) * (size_t)n * n);
        if (po_weights(n, seqs, lens, wf) != 0) {
            free(wf);
            po_destroy(p);
            return NULL;
        }
        for (int i = 0; i < n * n; i++) p->w[i] = (int32_t)wf[i]; /* (int) truncation, Node.cpp:226 */
        free(wf);
    }
    return p;
}

void po_destroy(po_problem *p)
{
    if (!p) return;
    for (int i = 0; i < p->n; i++) free(p->seq[i]);
    for (int k = 0; k < p->npairs; k++) free(p->table[k]);
    free(p);
}

const int32_t *po_table(const po_problem *p, int pair, int *rows, int *cols)
{
    *rows = p->len[p->pa[pair]] + 1;
    *cols = p->len[p->pb[pair]] + 1;
    return p->table[pair];
}
const int32_t *po_int_weights(const po_problem *p) { return p->w; }

int32_t po_calculate_h(const po_problem *p, const uint16_t *pos) /* HeuristicHPair.cpp:73-86 */
{
    int32_t h = 0;
    for (int k = 0; k < p->npairs; k++) {
        int x = p->pa[k], y = p->pb[k];
        h += p->table[k][(size_t)pos[x] * (p->len[y] + 1) + pos[y]] * p->w[x * p->n + y];
    }
    return h;
}

/* ------------------------------------------------------------------------ */
/* Owner hashes — CoordHash.cpp                                              */
/* ------------------------------------------------------------------------ */
static uint32_t zorder_hash(int n, const uint16_t *c, int shift, int size) /* :105-134 (n=N) and :137-166 (n=2) */
{
    int hash = 0;
    int bit_to_read = shift / n;
    unsigned int bits = (unsigned int)(log2((double)size) + (shift % n) + 1);
    unsigned int total = 1u << bits;
    if (total == 0) total = UINT_MAX;
    for (unsigned int bit_to_write = 1; bit_to_write <= total;) {
        for (unsigned int j = 0; j < (unsigned int)n && bit_to_write <= total; ++j) {
            if (bit_to_read < 31 && (c[j] & (1 << bit_to_read))) hash |= bit_to_write;
            bit_to_write <<= 1;
        }
        ++bit_to_read;
    }
    return (uint32_t)((hash >> (shift % n)) % size);
}

uint32_t po_owner(int n, const uint16_t *c, int hash_type, int shift, int size)
{
    if (shift < 0 || shift > 21) return UINT32_MAX; /* :241 throws invalid_argument */
    unsigned int sum = 0;
    switch (hash_type) {
    case PO_HASH_FSUM: /* :27-44 */
        for (int i = 0; i < n; i++) sum += c[i];
        return (sum >> shift) % size;
    case PO_HASH_PSUM: /* :47-61 */
        return ((unsigned int)(c[0] + c[1]) >> shift) % size;
    case PO_HASH_PZORDER:
        return zorder_hash(2, c, shift, size);
    default:
        return zorder_hash(n, c, shift, size);
    }
}

/* ------------------------------------------------------------------------ */
/* Successor expansion — Node.cpp:69-77,129-152,205-248; Coord.cpp:92-106    */
/* ------------------------------------------------------------------------ */
static int pair_cost(int neigh_num, int parenti, int mm_cost, int s1, int s2) /* Node.cpp:129-152 */
{
    int s;
    if ((neigh_num & (1 << s1)) && (neigh_num & (1 << s2))) return mm_cost;
    if (neigh_num & (1 << s1))
        s = s2;
    else if (neigh_num & (1 << s2))
        s = s1;
    else
        return PO_GAP_GAP;
    if (((parenti & (1 << s)) != 0) != ((neigh_num & (1 << s)) != 0)) return PO_GAP_OPEN;
    return PO_GAP_EXTENSION;
}

int po_get_neigh(const po_problem *p, const uint16_t *pos, int32_t g, int32_t parenti, int vec_size, int hash_type,
                 int shift, po_succ *out)
{
    int n = p->n, np = p->npairs;
    int mm[PO_MAX_SEQ * PO_MAX_SEQ];
    for (int k = 0; k < np; k++) /* Node.cpp:221-231; seq[len] is the NUL terminator (F14) */
        mm[k] = po_cost((unsigned char)p->seq[p->pa[k]][pos[p->pa[k]]], (unsigned char)p->seq[p->pb[k]][pos[p->pb[k]]]);
    int total = (1 << n) - 1;
    po_succ *tmp = (po_succ *)malloc(sizeof(po_succ) * (size_t)total);
    int cnt = 0;
    for (int i = 1; i <= total; i++) {
        po_succ s;
        memset(&s, 0, sizeof(s));
        int ok = 1;
        for (int d = 0; d < n; d++) { /* Coord.cpp:92-106 + Node.cpp:69-77 */
            s.pos[d] = (uint16_t)(pos[d] + ((i >> d) & 1));
            if (s.pos[d] > p->len[d]) ok = 0;
        }
        if (!ok) continue;
        int costs = 0;
        for (int k = 0; k < np; k++) costs += pair_cost(i, parenti, mm[k], p->pa[k], p->pb[k]) * p->w[p->pa[k] * n + p->pb[k]];
        s.g = g + costs;
        s.f = s.g + po_calculate_h(p, s.pos); /* Node.cpp:32-39 */
        s.parenti = i;
        s.owner = po_owner(n, s.pos, hash_type, shift, vec_size);
        tmp[cnt++] = s;
    }
    /* reference order: bucket by owner, ascending mask inside (Node.cpp:244) */
    int o = 0;
    for (int b = 0; b < vec_size; b++)
        for (int k = 0; k < cnt; k++)
            if ((int)tmp[k].owner == b) out[o++] = tmp[k];
    free(tmp);
    return o;
}

/* ------------------------------------------------------------------------ */
/* Serial A* — AStar.cpp:53-104, PriorityList.h:84-122                       */
/* ------------------------------------------------------------------------ */
typedef struct {
    uint16_t pos[PO_MAX_SEQ];
    int32_t g, f, parenti;
    int8_t state; /* 0 empty, 1 open, 2 closed */
    uint32_t stamp; /* version of the live heap entry */
} anode;

typedef struct {
    int32_t f;
    uint32_t stamp;
    uint64_t seqno;
    uint32_t slot;
} hent;

typedef struct {
    anode *tab;
    uint64_t cap, used;
    hent *heap;
    uint64_t hn, hcap, seqno;
    int n;
} astar;

static uint64_t pos_hash(const uint16_t *pos, int n)
{
    uint64_t h = 1469598103934665603ull;
    for (int i = 0; i < n; i++) {
        h ^= pos[i];
        h *= 1099511628211ull;
    }
    h ^= h >> 29;
    return h;
}

static void tab_grow(astar *a);

static uint32_t tab_find(astar *a, const uint16_t *pos, int create)
{
    if (create && (a->used + 1) * 10 > a->cap * 7) tab_grow(a);
    uint64_t i = pos_hash(pos, a->n) & (a->cap - 1);
    for (;;) {
        anode *e = &a->tab[i];
        if (e->state == 0) {
            if (!create) return UINT32_MAX;
            memcpy(e->pos, pos, sizeof(uint16_t) * a->n);
            a->used++;
            return (uint32_t)i;
        }
        if (memcmp(e->pos, pos, sizeof(uint16_t) * a->n) == 0) return (uint32_t)i;
        i = (i + 1) & (a->cap - 1);
    }
}

static void heap_push(astar *a, hent e)
{
    if (a->hn == a->hcap) {
        a->hcap *= 2;
        a->heap = (hent *)realloc(a->heap, sizeof(hent) * a->hcap);
    }
    uint64_t i = a->hn++;
    while (i > 0) {
        uint64_t par = (i - 1) / 2;
        hent *q = &a->heap[par];
        if (q->f < e.f || (q->f == e.f && q->seqno < e.seqno)) break;
        a->heap[i] = *q;
        i = par;
    }
    a->heap[i] = e;
}

static hent heap_pop(astar *a)
{
    hent top = a->heap[0];
    hent e = a->heap[--a->hn];
    uint64_t i = 0;
    for (;;) {
        uint64_t l = 2 * i + 1, r = l + 1, m = l;
        if (l >= a->hn) break;
        if (r < a->hn && (a->heap[r].f < a->heap[l].f || (a->heap[r].f == a->heap[l].f && a->heap[r].seqno < a->heap[l].seqno)))
            m = r;
        if (e.f < a->heap[m].f || (e.f == a->heap[m].f && e.seqno < a->heap[m].seqno)) break;
        a->heap[i] = a->heap[m];
        i = m;
    }
    if (a->hn) a->heap[i] = e;
    return top;
}

static void tab_grow(astar *a)
{
    anode *old = a->tab;
    uint64_t oc = a->cap;
    a->cap *= 2;
    a->tab = (anode *)calloc(a->cap, sizeof(anode));
    a->used = 0;
    /* slots move: rebuild the heap's slot references */
    uint32_t *remap = (uint32_t *)malloc(sizeof(uint32_t) * oc);
    for (uint64_t i = 0; i < oc; i++) {
        remap[i] = UINT32_MAX;
        if (old[i].state) {
            uint32_t s = tab_find(a, old[i].pos, 1);
            a->tab[s] = old[i];
            remap[i] = s;
        }
    }
    for (uint64_t i = 0; i < a->hn; i++) a->heap[i].slot = remap[a->heap[i].slot];
    free(remap);
    free(old);
}

/* PriorityList.h:104-113 */
static void open_conditional_enqueue(astar *a, const uint16_t *pos, int32_t g, int32_t f, int32_t parenti)
{
    uint32_t s = tab_find(a, pos, 1);
    anode *e = &a->tab[s];
    if (e->state == 1 && f >= e->f) return;
    e->g = g;
    e->f = f;
    e->parenti = parenti;
    e->state = 1;
    e->stamp++;
    hent h = {f, e->stamp, a->seqno++, s};
    heap_push(a, h);
}

/* The search loop of po_astar: runs until the goal is popped, the open list empties or `budget` pops, and leaves the
 * table and heap in *a for the caller to read and free. */
static void astar_run(const po_problem *p, int64_t budget, po_search_result *res, astar *out)
{
    int n = p->n;
    astar a;
    memset(&a, 0, sizeof(a));
    a.n = n;
    a.cap = 1 << 16;
    a.tab = (anode *)calloc(a.cap, sizeof(anode));
    a.hcap = 1 << 16;
    a.heap = (hent *)malloc(sizeof(hent) * a.hcap);
    memset(res, 0, sizeof(*res));
    res->g = res->f = -1;
    uint16_t zero[PO_MAX_SEQ] = {0}, fin[PO_MAX_SEQ] = {0};
    for (int i = 0; i < n; i++) fin[i] = (uint16_t)p->len[i];
    /* Sequences.cpp:70-77: initial node, parenti = all ones */
    open_conditional_enqueue(&a, zero, 0, po_calculate_h(p, zero), (1 << n) - 1);
    po_succ *succ = (po_succ *)malloc(sizeof(po_succ) * (size_t)((1 << n) - 1));
    int64_t open_live = 1;
    while (a.hn) {
        hent top = heap_pop(&a);
        anode *cur = &a.tab[top.slot];
        if (cur->state != 1 || cur->stamp != top.stamp) continue; /* superseded heap entry */
        /* AStar.cpp:69-80: the open list is pos-unique and a successor that
           beats a closed node erases it, so a dequeued node is never in CLOSED */
        res->pops++;
        open_live--;
        cur->state = 2;
        res->closed_size++;
        if (memcmp(cur->pos, fin, sizeof(uint16_t) * n) == 0) {
            res->finished = 1;
            res->g = cur->g;
            res->f = cur->f;
            break;
        }
        res->expansions++;
        uint16_t cpos[PO_MAX_SEQ];
        memcpy(cpos, cur->pos, sizeof(cpos));
        int32_t cg = cur->g, cpar = cur->parenti;
        int cnt = po_get_neigh(p, cpos, cg, cpar, 1, PO_HASH_FZORDER, 12, succ);
        res->generated += cnt;
        for (int k = 0; k < cnt; k++) {
            uint32_t s = tab_find(&a, succ[k].pos, 0);
            if (s != UINT32_MAX && a.tab[s].state == 2) { /* AStar.cpp:86-91 */
                if (succ[k].g >= a.tab[s].g) continue;
                a.tab[s].state = 0 + 3; /* erased from CLOSED; slot stays claimed */
                res->closed_size--;
                res->reopen++;
            }
            int was_open = (s != UINT32_MAX && a.tab[s].state == 1);
            open_conditional_enqueue(&a, succ[k].pos, succ[k].g, succ[k].f, succ[k].parenti);
            if (!was_open) open_live++;
        }
        if (budget > 0 && res->pops >= budget) break;
    }
    res->open_size = open_live;
    free(succ);
    *out = a;
}

int po_astar(const po_problem *p, int64_t budget, po_search_result *res, char **rows)
{
    int n = p->n;
    uint16_t fin[PO_MAX_SEQ] = {0};
    for (int i = 0; i < n; i++) fin[i] = (uint16_t)p->len[i];
    astar a;
    astar_run(p, budget, res, &a);
    if (res->finished && rows) {
        /* backtrace.cpp:44-69 */
        int total = 0;
        for (int i = 0; i < n; i++) total += p->len[i];
        char *buf = (char *)malloc((size_t)n * (total + 1));
        int cols = 0;
        uint16_t cp[PO_MAX_SEQ];
        memcpy(cp, fin, sizeof(cp));
        for (;;) {
            int allz = 1;
            for (int i = 0; i < n; i++)
                if (cp[i]) allz = 0;
            if (allz) break;
            anode *e = &a.tab[tab_find(&a, cp, 0)];
            for (int i = 0; i < n; i++) {
                int moved = (e->parenti >> i) & 1;
                buf[(size_t)i * (total + 1) + cols] = moved ? p->seq[i][cp[i] - 1] : '-';
                if (moved) cp[i]--;
            }
            cols++;
        }
        for (int i = 0; i < n; i++) {
            for (int c = 0; c < cols; c++) rows[i][c] = buf[(size_t)i * (total + 1) + (cols - 1 - c)];
            rows[i][cols] = 0;
        }
        free(buf);
    }
    free(a.tab);
    free(a.heap);
    return 0;
}

int64_t po_astar_settled(const po_problem *p, int64_t budget, int64_t cap, int32_t *F_out, uint16_t *pos, int32_t *g,
                         int32_t *parenti, po_search_result *res)
{
    int n = p->n;
    astar a;
    astar_run(p, budget, res, &a);
    int32_t F = INT32_MAX;
    for (uint64_t i = 0; i < a.hn; i++) { /* the best live entry: skip superseded ones */
        const anode *e = &a.tab[a.heap[i].slot];
        if (e->state == 1 && e->stamp == a.heap[i].stamp && a.heap[i].f < F) F = a.heap[i].f;
    }
    *F_out = F;
    int64_t k = 0;
    for (uint64_t i = 0; i < a.cap; i++) {
        const anode *e = &a.tab[i];
        if (e->state != 2 || e->f >= F) continue;
        if (k < cap) {
            memcpy(pos + (size_t)k * n, e->pos, sizeof(uint16_t) * n);
            g[k] = e->g;
            parenti[k] = e->parenti;
        }
        k++;
    }
    free(a.tab);
    free(a.heap);
    return k;
}
