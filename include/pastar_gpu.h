/*
 * pastar_gpu.h — C ABI of the B200-native PA-Star data-parallel core.
 *
 * The reference (Gabrielcarvfer/mpi_pastar_msa) has no FFI seam: its hot path
 * is reached through C++ template classes and three singletons.  This header
 * is the boundary a maintainer binds instead; every entry point names the
 * reference interface it replaces (paths relative to the reference root).
 * INTEGRATION.md shows the reference-side shim for each.
 *
 * Conventions
 *   - every call returns a pg_status (0 = ok); no exception crosses the ABI;
 *     pg_last_error(ctx) gives the message of the last failure.
 *   - plain pointers and sizes only.  Entry points ending in _dev take DEVICE
 *     pointers (and a cudaStream_t passed as void*); all others take HOST
 *     pointers and do their own host<->device copies.
 *   - there is no CPU fallback: without a CUDA device pg_ctx_create fails
 *     with PG_ERR_CUDA.
 *   - a context is bound to one device and is not thread-safe; use one
 *     context per host thread / per GPU.
 *
 * Record layouts (binary compatible with the reference)
 *   pg_node  = Node<N>   : uint16 pos[N]; pad to 4; int32 f; int32 g; int32 parenti
 *              (pastar/include/Node.h:28-49, Coord.h:68; sizes in SURVEY F7)
 *   pg_succ  = pg_node + uint32 owner            (owner = Coord<N>::get_id(vec_size))
 *   Strides: pg_node_stride(N) = ((2N+3)&~3)+12, pg_succ_stride(N) = that + 4.
 */
#ifndef PASTAR_GPU_H
#define PASTAR_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_MAX_SEQ 16
#define PG_ABI_VERSION 1

typedef enum {
    PG_OK = 0,
    PG_ERR_ARG = 1,         /* bad argument (null, N unsupported, ...)                         */
    PG_ERR_CUDA = 2,        /* CUDA runtime failure, or no device                              */
    PG_ERR_UNSUPPORTED = 3, /* problem outside the supported domain (packed key > 128 bits)    */
    PG_ERR_CAPACITY = 4,    /* closed/open table or open-list pool exhausted                   */
    PG_ERR_STATE = 5,       /* call out of order (e.g. expand before pg_build_pair_tables)     */
    PG_ERR_HASH_SHIFT = 6   /* hash shift outside 0..21: CoordHash.cpp:240-242 throws here     */
} pg_status;

/* hashType, pastar/include/Coord.h:28 (same numeric values) */
typedef enum { PG_HASH_FZORDER = 0, PG_HASH_PZORDER = 1, PG_HASH_FSUM = 2, PG_HASH_PSUM = 3 } pg_hash_type;

typedef struct pg_ctx pg_ctx;

static inline int pg_node_stride(int n) { return ((2 * n + 3) & ~3) + 12; }
static inline int pg_succ_stride(int n) { return ((2 * n + 3) & ~3) + 16; }

/* ------------------------------------------------------------------ host-side producers */

/* Replaces Cost::Cost / Cost::cost (pastar/Cost.cpp:12-271, include/Cost.h:13,49):
 * writes the 90x90 PAM250-as-cost table (raw-ASCII indexed, unset pairs 0). */
void pg_default_cost_table(int32_t out90x90[90 * 90]);

/* Replaces weightAltschulsRationale2 (pastar/WeightedSP.cpp:424-519): float pair
 * weights, n x n row-major, float-operation-for-float-operation equal to the
 * reference.  Host code (serial, float-order sensitive; the reference keeps it
 * on the host too).  Unlike the reference (fixed 1000x1000 scratch, heap
 * overflow at L >= 999) any length is accepted. */
int pg_host_weights(int n_seq, const char *const *seqs, const int *lens, float *w_out);

/* The same weights with the pair loop (the reference's `primer`: N(N-1)/2 three-matrix forward alignments and their
 * tracebacks, pastar/WeightedSP.cpp:144-244, 109-142 - half of HeuristicHPair::init) run as ONE kernel on `device`
 * (< 0: the current one); the neighbour-joining tree and the float propagation (WeightedSP.cpp:317-420, 464-509) stay on
 * the host.  Output bit-identical to pg_host_weights.  kernel_ms (may be NULL) receives the kernel's CUDA-event time.
 * PG_ERR_UNSUPPORTED when a sequence is too long for the shared-memory sweep (about 5 800 residues): use pg_host_weights. */
int pg_gpu_weights(int n_seq, const char *const *seqs, const int *lens, int device, float *w_out, float *kernel_ms);

/* ------------------------------------------------------------------ context */

/* Replaces Sequences::set_seq + the Cost/HeuristicHPair singletons' state
 * (pastar/Sequences.cpp:39-51, include/Sequences.h:19-28).  Uploads residues,
 * cost table (NULL = pg_default_cost_table), gap constants (Cost.h:13: 30/30/30)
 * and the truncated pair weights (int)weightMatrix[i][j] (n x n, NULL = all 1).
 * device < 0 keeps the current CUDA device. */
int pg_ctx_create(int n_seq, const char *const *seqs, const int *lens, const int32_t *cost90x90, int gap_open,
                  int gap_ext, int gap_gap, const int32_t *w_int, int device, pg_ctx **out);
/* The reference instantiates its templates for N in {3..10, 14, 16} only (pastar/include/max_seq_helper.h:9-19) and
 * pg_ctx_create follows it.  pg_allow_extended_n(1) - an explicit, process-wide opt-in that diverges from the reference -
 * also admits N = 11, 12, 13, 15 (pairwise tables, weights, getNeigh batches and the one-GPU search; the partitioned
 * search is not built for them and pg_search_begin refuses n_parts > 1). */
int pg_allow_extended_n(int enable);
void pg_ctx_destroy(pg_ctx *ctx);
const char *pg_last_error(const pg_ctx *ctx);
int pg_abi_version(void);
/* Measurement helper: random 16-byte loads per second over a `bytes`-sized table (8 in flight per thread): the
 * measured hardware ceiling for the closed/open-table probe, reported by bench.py next to the kernel's rate. */
int pg_bench_random_gather(int device, int64_t bytes, double *loads_per_sec);
/* Measurement helper: DP-cell instruction groups (3 adds + one 3-input minimum, 8 independent chains per thread) per
 * second on all SMs: the measured integer peak the pairwise-DP GCUPS are compared with. */
int pg_bench_int_peak(int device, double *cells_per_sec);
/* Run every later launch of this context on the caller's stream (cudaStream_t as void*; NULL = the legacy
 * default stream as everywhere in CUDA, (void*)-1 = back to the context's own non-blocking stream), e.g. torch's
 * current stream so that the caller's CUDA events bracket the work and NCCL collectives are ordered with it. */
int pg_ctx_set_stream(pg_ctx *ctx, void *stream);

/* ------------------------------------------------------------------ (1) pairwise DP heuristic */

/* Replaces the PairAlign loop of HeuristicHPair::init (pastar/HeuristicHPair.cpp:47-61
 * -> PairAlign.cpp:137-171): all N(N-1)/2 reverse DP tables in one launch,
 * left device-resident.  kernel_ms (may be NULL) receives the CUDA-event time. */
int pg_build_pair_tables(pg_ctx *ctx, float *kernel_ms);
/* PairAlign::getScore (PairAlign.cpp:174-177) for a whole table: rows x cols int32, row-major. */
int pg_pair_table_shape(const pg_ctx *ctx, int pair, int *rows, int *cols);
int pg_copy_pair_table(pg_ctx *ctx, int pair, int32_t *out);
/* HeuristicHPair::calculate_h<N> (HeuristicHPair.cpp:73-86) for n coords (n x N uint16). */
int pg_calculate_h(pg_ctx *ctx, const uint16_t *coords, int64_t n, int32_t *out);

/* ------------------------------------------------------------------ (3) owner hash */

/* Coord<N>::configure_hash (pastar/CoordHash.cpp:260-265); default FZORDER / 12. */
int pg_configure_hash(pg_ctx *ctx, int hash_type, int hash_shift);
/* Coord<N>::get_id(size) (CoordHash.cpp:190-245) for n coords. */
int pg_owner(pg_ctx *ctx, const uint16_t *coords, int64_t n, int size, uint32_t *out);

/* ------------------------------------------------------------------ (2) batched expansion */

/* Replaces Node<N>::getNeigh (pastar/Node.cpp:205-248) for k parents at once.
 * parents: k records in pg_node layout (== Node<N>).  out_succ: room for
 * k * (2^N - 1) records in pg_succ layout; parent i's successors start at
 * record i * (2^N - 1), in ascending move-mask order, out_counts[i] of them
 * (borderCheck-failing masks are not emitted, as in the reference). */
int pg_expand_batch(pg_ctx *ctx, const void *parents, int64_t k, int vec_size, void *out_succ, int32_t *out_counts);
int pg_expand_batch_dev(pg_ctx *ctx, const void *d_parents, int64_t k, int vec_size, void *d_out_succ,
                        int32_t *d_out_counts, void *stream);

/* ------------------------------------------------------------------ (3)+(4) search */

typedef struct {
    int32_t n_parts;        /* number of hash-owned partitions (= GPUs); 1 = single GPU          */
    int32_t part;           /* this context's partition id                                       */
    int64_t table_capacity; /* closed+open table slots (rounded up to a power of two); 0 = auto  */
    int64_t batch_target;   /* frontier nodes popped per round (whole f-buckets, at least one); 0 = auto */
    int64_t max_expansions; /* > 0: stop after this many expansions (budgeted run, not optimal)  */
    int32_t rounds_per_sync;/* rounds launched between host checks; 0 = auto                     */
    int32_t reserved;       /* 1 = P2P successor records, 2 = P2P parent forwarding: see pg_search_set_peers */
} pg_search_config;

typedef struct {
    int32_t finished;       /* 1 = optimal goal reached; 0 = budget hit                          */
    int32_t g, f;           /* "Final Score" g and f (Node.cpp:41-47)                            */
    int32_t align_len;      /* columns of the alignment                                          */
    int64_t pops;           /* dequeues incl. stale ones: the reference's "Total" (PAStar.cpp:341) */
    int64_t expansions;     /* nodes run through the getNeigh-equivalent                         */
    int64_t generated;      /* successors produced (after borderCheck)                           */
    int64_t reopen;         /* PAStar.cpp:231,347                                                */
    int64_t open_size, closed_size;
    int64_t rounds;
    int64_t probed;         /* successors looked up in the closed/open table (generated - pruned) */
    int64_t pushed;         /* successors that were new or strictly better: pushed to the open list */
    int64_t inserted;       /* distinct coordinates in the table                                  */
    double seconds;         /* phase-2 wall time                                                 */
    double kernel_ms;       /* CUDA-event time from the first to the last round of the search     */
    double expand_ms;       /* sum of the fused expand kernel's launch durations (profiling on)  */
    double select_ms;       /* sum of the select kernel's launch durations (profiling on)        */
    double claim_ms;        /* ... of the claim kernel (closed-bit claim + compaction of live parents) */
    double insert_ms;       /* ... of the insert kernel over the round's local survivors          */
    int64_t survivors;      /* records run through the insert kernel (local survivors + received records) */
    double inbox_ms;        /* ... of the insert kernels over the records received from other partitions (P2P mode) */
} pg_result;

/* Replaces PAStar<N>::pa_star (pastar/PAStar.cpp:626-673) on ONE GPU
 * (cfg->n_parts must be 1): batched pop -> expand -> dedupe -> push until the
 * optimality-preserving stop (PAStar.cpp:410-547: goal accepted only when no
 * open node has f < g_goal).  rows (may be NULL): N buffers of at least
 * sum(lens)+1 bytes receive the aligned sequences (backtrace.cpp:77-109). */
int pg_search(pg_ctx *ctx, const pg_search_config *cfg, pg_result *res, char *const *rows);

/* The same search hash-partitioned over n_gpus GPUs of one box, driven by ONE host process: ctxs[i] is a context
 * created on device i (same sequences, weights and hash configuration; pair tables built).  Replaces pa_star with
 * threads x MPI ranks (PAStar.cpp:626-673), the sender / receiver / decoder threads (pastar_functions/*.cpp) and
 * check_stop's allreduces (PAStar.cpp:502-519): one partition per GPU (owner = Coord::get_id(n_gpus)), parent
 * forwarding over peer-mapped inboxes (NVLink), cross-GPU ordering by stream-wait events, no NCCL.  total = summed
 * counters + final score + alignment rows; parts (may be NULL) = n_gpus per-partition counters (the reference's
 * per-thread rows of "Total nodes count:").  cfg->n_parts / part / reserved are ignored. */
int pg_multi_search(pg_ctx *const *ctxs, int n_gpus, const pg_search_config *cfg, pg_result *total, pg_result *parts,
                    char *const *rows);

/* Step-wise form for hash-partitioned multi-GPU drivers (one context per GPU,
 * the exchange between the two calls is the driver's: NCCL all-to-all).
 * Replaces worker_inner's expand + reconciliation (PAStar.cpp:319-401) and
 * sender/receiver (pastar_functions/PAStarSender.cpp, PAStarReceiver.cpp). */
int pg_search_begin(pg_ctx *ctx, const pg_search_config *cfg);
/* Pop up to batch_target nodes whose f < f_limit and expand them; successors
 * owned by this partition are deduped and pushed, the others are appended to
 * per-destination outboxes as pg_xrec records. */
int pg_search_round(pg_ctx *ctx, int32_t f_limit);
/* `rounds` rounds back to back with one host synchronisation at the end (single partition only). */
int pg_search_rounds(pg_ctx *ctx, int32_t rounds, int32_t f_limit);
/* Per-launch CUDA-event timing of the select and expand kernels (off by default: two event records per launch). */
int pg_search_profile(pg_ctx *ctx, int enable);
/* Device-driven P2P rounds (pg_search_round_async + pg_search_insert_inbox_async) take the same arguments every second
 * round, so a caller may capture an even number of them into a CUDA graph on the context's stream and replay it.  The
 * library's own round counter (pg_result.rounds / pg_search_status) only sees the calls it executes: `delta` adds the
 * replayed rounds (or takes back the ones that were captured, not run). */
int pg_search_note_rounds(pg_ctx *ctx, int64_t delta);
/* The large device buffers of a search (value blocks, directory, open-list pool, survivor list) are kept by the library
 * when a search ends and reused by the next search of the same size on the same device (PAStar.cpp:626-673 allocates
 * per run; here a 16 GiB cudaMalloc + cudaFree costs more than a small search).  This gives them back to the driver. */
void pg_release_cached_memory(void);
/* Device pointer + record count of the outbox for partition dst (valid until the next round). */
int pg_search_outbox(pg_ctx *ctx, int dst, void **d_records, int64_t *count);
/* P2P mode (the fused compute + exchange variant): give every partition's inbox base as seen from THIS device
 * (peer-mapped over NVLink, e.g. torch symmetric memory / CUDA IPC).  The expand kernel then stores remote
 * successors straight into region [part] of inbox[dst] (pg_search_outbox_capacity() records of pg_xrec_stride()
 * bytes per region) while it computes; only the per-destination counts still travel by collective.  Request it
 * with pg_search_config.reserved = 1 in pg_search_begin (no local outbox is allocated). */
int pg_search_set_peers(pg_ctx *ctx, void *const *peer_inbox, int n);
/* Device-driven P2P rounds (no host round trip, no collective for the counts): peer_counts[r] is partition r's
 * uint64[nbuf][n_parts] array as seen from this device.  After its expand kernel a partition stores "records I
 * wrote into your inbox" at peer_counts[dst][buf][part]; the driver then runs one cross-GPU barrier on the stream
 * and calls pg_search_insert_inbox_async, whose insert kernels read the counts from device memory.  With nbuf = 2
 * the inboxes (2 x n_parts regions) and count arrays alternate per round, so that one barrier per round is enough. */
int pg_search_set_peer_counts(pg_ctx *ctx, void *const *peer_counts, int n, int nbuf);
/* Data-flow synchronisation instead of a barrier (needs nbuf = 2): every count a partition publishes carries the exchange
 * round, and pg_search_insert_inbox_async starts with a one-block kernel that waits, on the device, until every source's
 * count of the current round has arrived.  The driver then calls pg_search_round_async / pg_search_insert_inbox_async
 * back to back with NO cross-GPU barrier in between: a count is written after the data it covers, and no partition can
 * run more than one round ahead of another (its next round waits for that partition's next count).  A peer that never
 * delivers ends the wait after ~20 s with PG_ERR_STATE. */
int pg_search_set_device_sync(pg_ctx *ctx, int enable);
/* pg_search_round without the host synchronisation (launches only); pair with pg_search_sync. */
int pg_search_round_async(pg_ctx *ctx, int32_t f_limit);
int pg_search_insert_inbox_async(pg_ctx *ctx);
/* bytes one source partition may write into one inbox per buffer: the symmetric allocation the driver makes is
 * nbuf x n_parts x this.  pg_search_config.reserved selects what crosses NVLink: 1 = successor records
 * (pg_xrec), stored by the expand kernel; 2 = parent forwarding: the claim kernel sends each live parent
 * (key + g + parenti, 16 or 24 bytes) to every partition that owns one of its successors, and that partition
 * generates them itself - about fifty times less traffic for the same result. */
int64_t pg_search_region_bytes(const pg_ctx *ctx);
/* wait for the launched rounds; reports capacity errors like pg_search_round */
int pg_search_sync(pg_ctx *ctx);
int64_t pg_search_outbox_capacity(const pg_ctx *ctx);
/* device pointer to the per-destination record counts of the last round (uint64[64]) */
int pg_search_outbox_counts_dev(pg_ctx *ctx, void **d_counts);
/* insert n segments: segment i = counts[i] records at base + i*stride_bytes (one host sync at the end) */
int pg_search_insert_segments_dev(pg_ctx *ctx, const void *base, int64_t stride_bytes, const int64_t *counts, int n);
/* Dedupe + push records received from other partitions (device pointer). */
int pg_search_insert_dev(pg_ctx *ctx, const void *d_records, int64_t count);
/* Local lower bound of open f (INT32_MAX when empty), best goal g seen here
 * (INT32_MAX when none) and counters so far. */
int pg_search_status(pg_ctx *ctx, int32_t *min_open_f, int32_t *best_goal_g, pg_result *counters);
/* Closed/open table lookup for the distributed backtrace
 * (pastar_functions/PAStarDistributedBacktrace.cpp:18-214): found=0 if absent. */
int pg_search_lookup(pg_ctx *ctx, const uint16_t *pos, int32_t *found, int32_t *g, int32_t *parenti);
/* The same lookup for `count` coordinates (host arrays; pos is count x N): state[i] 0 absent, 1 open, 2 closed; g[i] and
 * parenti[i] are -1 when absent.  One device thread per coordinate; no project counterpart (it serves table checks).
 * PG_ERR_ARG, before any device work, when a position is past its sequence's length or no search is active. */
int pg_search_lookup_batch(pg_ctx *ctx, const uint16_t *pos, int64_t count, int32_t *state, int32_t *g, int32_t *parenti);
int pg_search_end(pg_ctx *ctx);
/* Bounded-suboptimal (weighted) search - an opt-in extension of pg_search / pg_multi_search / pg_search_begin (the
 * reference, PAStar.cpp:626-673, only searches for the optimum).  Every later search on the context orders, prunes and
 * stops on f_w = g + h_w, h_w = sum over pairs of floor(num * w_ij * T_ij / den), h <= h_w <= (num/den) h, and returns an
 * alignment that costs at most num/den times the optimum.  den is a power of two in 1..1024, den <= num <= 16 den;
 * (1, 1), the default, is the exact search and leaves every result unchanged.  pg_expand_batch and pg_calculate_h stay
 * unweighted.  With num > den the reported g = f is the re-scored cost of the alignment returned (its parent chain may be
 * cheaper than the best goal found).  PG_ERR_ARG for a bad weight, PG_ERR_STATE while a step-wise search is active;
 * pg_multi_search refuses contexts whose weights differ (PG_ERR_ARG), and pg_search_begin refuses, with
 * PG_ERR_UNSUPPORTED, a weighted f range beyond 2^27 buckets. */
int pg_search_set_weight(pg_ctx *ctx, int32_t num, int32_t den);
/* Certified lower bound on the optimal cost: the minimum of g + h over the open entries, of g + h over the successors a
 * weighted search dropped, of the best goal and of the all-advance cost.  After pg_search / pg_multi_search: the bound of
 * that search (every context of a pg_multi_search reports the global one); a finished search has g * den <= num * bound
 * (an exact search: bound == g), a budgeted one bound <= optimum.  While a step-wise search is active: this partition's
 * bound, computed now (the driver takes the minimum over the partitions between rounds).  PG_ERR_STATE before any
 * search. */
int pg_search_lower_bound(pg_ctx *ctx, int32_t *lower_bound);
/* Cost of an alignment under the context's cost model (the arithmetic of the search's g; host code, O(cols * pairs)).
 * rows: N NUL-terminated rows of exactly `cols` characters; each row with its '-' removed must spell the context's
 * sequence and no column may hold gaps only.  PG_ERR_ARG with a message otherwise.  Needs no device. */
int pg_score_alignment(pg_ctx *ctx, const char *const *rows, int32_t cols, int64_t *cost);
/* Incumbent-bounded search - an opt-in extension of pg_search / pg_multi_search / pg_search_begin (the reference only
 * searches from scratch; Ikeda & Imai 1999's "enhanced A*").  Scores `rows` (as pg_score_alignment), keeps a copy and
 * makes its cost U the upper bound of every later search on the context: an exact search keeps only successors with
 * g + h < U, a weighted one those with g + floor(h_w * floor(2^32 / weight) / 2^32) < U (a value <= g + h), and goals
 * need g < U.  The bucket range, prune and goal limits and the value width follow from U.  Results:
 *   finished = 1: a cheaper alignment, with its rows and cost;
 *   finished = 2: the search ran out of nodes below U (or h(start) >= U): the incumbent's rows and g = U are returned,
 *                 and an exact search then reports lower bound == U - a proof that the incumbent is optimal;
 *   finished = 0: the expansion budget ran out (lower bound <= optimum <= U).
 * The lower bound (pg_search_lower_bound) is also capped by U.  rows == NULL clears the incumbent.  PG_ERR_STATE while
 * a step-wise search is active; pg_multi_search refuses contexts whose incumbent costs differ (PG_ERR_ARG). */
int pg_search_set_incumbent(pg_ctx *ctx, const char *const *rows, int32_t cols);
/* Anytime search on one GPU (restarting weighted A*, Richter, Thayer & Ruml, ICAPS 2010): phase k is a fresh pg_search
 * at weight weight_num[k] / weight_den[k] (each as in pg_search_set_weight; n_phases in 1..64) whose incumbent is the
 * best alignment so far - the caller's incumbent, if one is set, for phase 0.  cfg->max_expansions (0: none) is the
 * budget over all phases.  The loop stops early once the best lower bound reaches the incumbent's cost, when a phase
 * stops at the budget, or when a phase after the first runs out of table (PG_ERR_CAPACITY, kept as pg_last_error; the
 * best alignment so far is returned).  res: counters summed over the phases, g and the rows (may be NULL) of the best alignment;
 * finished = 1 when that alignment is proved optimal (lower bound == g), 2 when it is returned with a gap, 0 when no
 * alignment is known.  phase_res / phase_lb (may be NULL): each phase's result and lower bound; phases that did not
 * run are zeroed with phase_lb = -1.  Afterwards pg_search_lower_bound gives the maximum over the phases, the weight is
 * what it was before the call and the incumbent is the alignment returned. */
int pg_search_anytime(pg_ctx *ctx, const pg_search_config *cfg, const int32_t *weight_num, const int32_t *weight_den, int n_phases,
                      pg_result *res, pg_result *phase_res, int32_t *phase_lb, char *const *rows);
/* bytes per exchanged successor record for this context */
int pg_xrec_stride(const pg_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* PASTAR_GPU_H */
