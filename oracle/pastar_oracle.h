/* TEST INFRASTRUCTURE — CPU oracle for the PA-Star hot path.  Not shipped,
 * not linked by the product; only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load it.
 *
 * Plain-C restatement of the reference's algorithm (Gabrielcarvfer/
 * mpi_pastar_msa).  Every function cites the reference file:line it follows.
 *
 * PARITY PINNING: the reference ships no tests or golden vectors (SURVEY §4).
 * This oracle is pinned against the reference ITSELF: oracle/_ref/pastar_ref
 * is the unmodified reference arithmetic compiled in place (oracle/Makefile),
 * tests/test_oracle_vs_ref.py compares every function below with it on the
 * four FASTA fixtures and seeded random inputs, and tests/golden/ holds
 * fixtures generated from it (tests/golden/make_golden.py).
 */
#ifndef PASTAR_ORACLE_H
#define PASTAR_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { PO_HASH_FZORDER = 0, PO_HASH_PZORDER = 1, PO_HASH_FSUM = 2, PO_HASH_PSUM = 3 }; /* Coord.h:28 */
enum { PO_GAP_EXTENSION = 30, PO_GAP_OPEN = 30, PO_GAP_GAP = 30 };                     /* Cost.h:13 */
#define PO_MAX_SEQ 16

typedef struct po_problem po_problem;

typedef struct {
    uint16_t pos[PO_MAX_SEQ];
    int32_t f, g, parenti;
    uint32_t owner;
} po_succ;

typedef struct {
    int32_t finished, g, f;
    int64_t pops, expansions, generated, reopen, open_size, closed_size;
} po_search_result;

/* Cost.cpp:12-271: 90x90 int table indexed by raw ASCII. */
void po_cost_table(int32_t out[90 * 90]);
int po_cost(int a, int b);

/* PairAlign.cpp:137-171: reverse DP, row-major (l1+1) x (l2+1). */
void po_pair_table(const char *s1, int l1, const char *s2, int l2, int32_t *out);

/* WeightedSP.cpp:424-519: float pair weights, n x n row-major.  Returns 0, or
 * -1 when a sequence is longer than the reference's fixed scratch (F4). */
int po_weights(int n, const char *const *seqs, const int *lens, float *w_out);

/* Problem = sequences + P tables + truncated int weights
 * (HeuristicHPair.cpp:47-67).  w_int may be NULL: then po_weights is used. */
po_problem *po_create(int n, const char *const *seqs, const int *lens, const int32_t *w_int);
void po_destroy(po_problem *p);
const int32_t *po_table(const po_problem *p, int pair, int *rows, int *cols);
const int32_t *po_int_weights(const po_problem *p);

/* HeuristicHPair.cpp:73-86 */
int32_t po_calculate_h(const po_problem *p, const uint16_t *pos);

/* CoordHash.cpp:38-61,105-166,190-245; returns UINT32_MAX for shift > 21. */
uint32_t po_owner(int n, const uint16_t *pos, int hash_type, int shift, int size);

/* Node.cpp:205-248: all successors of one node, reference order (bucket by
 * owner, ascending mask inside a bucket).  Returns the count. */
int po_get_neigh(const po_problem *p, const uint16_t *pos, int32_t g, int32_t parenti, int vec_size, int hash_type,
                 int shift, po_succ *out);

/* AStar.cpp:53-104 with PriorityList.h:84-122 semantics; budget>0 stops after
 * that many pops.  rows (n strings of at least sum(lens)+1 bytes) may be NULL. */
int po_astar(const po_problem *p, int64_t budget, po_search_result *res, char **rows);

/* The settled set of the same search after `budget` pops (0: run to the goal).  *F_out receives the f of the best live
 * open entry (INT32_MAX when the open list is empty); every closed node with f < *F_out is written as pos[k * n ..],
 * g[k], parenti[k], the first `cap` of them.  Returns how many there are (more than cap: call again with more room).
 * Under a consistent heuristic these are exactly the nodes with g* + h < F, each with g == g*. */
int64_t po_astar_settled(const po_problem *p, int64_t budget, int64_t cap, int32_t *F_out, uint16_t *pos, int32_t *g,
                         int32_t *parenti, po_search_result *res);

#ifdef __cplusplus
}
#endif
#endif
