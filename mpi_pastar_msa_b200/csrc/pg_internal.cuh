// Internal declarations shared by the CUDA translation units of libpastar_gpu.
// sm_100a only; no other architecture is built and there is no CPU path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <climits>
#include <functional>
#include <string>
#include <vector>

#include "pastar_gpu.h"

#define PG_MAX_PAIRS (PG_MAX_SEQ * (PG_MAX_SEQ - 1) / 2)
#define PG_SM_COUNT_B200 148

// Device-side description of the problem, passed by value as a
// __grid_constant__ kernel parameter (about 3.3 KB, lives in the constant bank).
struct DevProblem {
    int n, npairs;
    int gap_open, gap_ext, gap_gap;
    int cell16;     // pairwise tables are uint16 (1) or int32 (0)
    int key_bits;   // bits per coordinate in the packed key
    int hash_type, hash_shift;
    int len[PG_MAX_SEQ];
    int w[PG_MAX_PAIRS];               // (int)weightMatrix[x][y] per pair, (i<j) order
    int cols[PG_MAX_PAIRS];            // row pitch of the pair's table in cells: len[y] + 1 rounded up to a multiple of 8
    uint8_t pa[PG_MAX_PAIRS], pb[PG_MAX_PAIRS]; // pair -> (x, y), x < y
    const uint8_t *seq[PG_MAX_SEQ];    // residues, len+1 bytes, trailing 0 (Node.cpp:225 reads seq[len])
    const void *table[PG_MAX_PAIRS];   // reverse DP tables, row-major (len[x]+1) x (len[y]+1)
    const int32_t *cost;               // 90 x 90
};

struct PairGeom {
    int a, b;       // sequence indices, a < b
    int rows, cols; // len+1
    int pitch;      // cells per stored row (cols rounded up to a multiple of 8: rows start 16-byte aligned)
    size_t offset;  // cell offset into the table arena
};

// ---- search state (pg_search.cu) -------------------------------------------------------------
struct SearchCtrl {          // lives in device memory; mirrored to pinned host memory on sync
    int32_t f0;              // bucket 0 corresponds to f == f0 (= h(start))
    int32_t f_range;         // number of buckets
    int32_t cursor;          // first bucket that may be non-empty
    int32_t best_goal;       // INT32_MAX until the goal has been generated
    int32_t prune_limit;     // successors with f >= this are dropped (upper bound + 1)
    int32_t done;            // 1 optimal, 2 open list exhausted
    int32_t error;           // 1 table full, 2 pool exhausted, 3 f beyond the bucket range, 4 outbox / survivor list overflow, 5 f below h(start)
    int32_t batch_n;         // parents selected for the current round
    int32_t plan_n;          // plan entries of the current round
    int32_t min_open_f;      // f of the first non-empty bucket after the last select (INT32_MAX if none)
    uint32_t chunk_bump;     // next free chunk
    int32_t drop_lb;         // weighted search: min over dropped successors of a value <= their g + h (INT32_MAX if none)
    unsigned long long pops, expansions, generated, reopen, inserted, pushed, pruned, table_used; // table_used: records seen by insert kernels
    unsigned long long surv_n;   // local survivors of the current round (records in SearchState::d_surv)
    unsigned long long live_n;   // live parents of the current round (after the closed-bit claim)
    unsigned long long xround;   // exchange rounds completed (device-driven P2P modes): the stamp of the counts is xround + 1, kept on
                                 // the device so that a round's launches take the same arguments every time (CUDA-graph replay)
    int free_top[16];            // open-list pool: chunks on the free stack of every size class (log2 units)
    unsigned long long phase[8]; // PG_PHASE_TIMING builds: warp-cycles per phase of the expand kernel
};

// Owner of an instantiated CUDA graph (a captured group of search rounds).
struct GraphExec {
    cudaGraphExec_t exec = nullptr;
    GraphExec() = default;
    GraphExec(const GraphExec &) = delete;
    GraphExec &operator=(const GraphExec &) = delete;
    ~GraphExec() { reset(); }
    void reset()
    {
        if (exec) cudaGraphExecDestroy(exec);
        exec = nullptr;
    }
    explicit operator bool() const { return exec != nullptr; }
};

struct PlanEntry;
struct SearchState {
    int keyw = 1;            // u64 words per packed key
    int valw = 8;            // bytes per value (4 when g, the open bit and the move mask fit 32 bits)
    int D = 0, DL = 0;       // block dimensions, directory-line dimensions
    int nb = 31, gs = 32;    // value layout: open bit, g shift
    uint64_t cap = 0;        // value slots = dir_slots << D (power of two)
    uint64_t dir_slots = 0;  // directory slots = blocks (power of two)
    unsigned long long *d_dir = nullptr;
    void *d_vals = nullptr;
    unsigned long long *d_buckets = nullptr;
    uint32_t *d_tail = nullptr;              // per bucket: entries in the chunks behind the head
    uint32_t *d_hint = nullptr;
    uint32_t *d_pool = nullptr;
    unsigned long long *d_link = nullptr;    // per unit: {offset, lg} of the previous chunk of the bucket
    uint32_t *d_free = nullptr;              // free stacks of popped chunks, one per size class
    uint32_t free_off[16] = {0};             // first entry of class lg's stack in d_free
    uint32_t n_units = 0;
    PlanEntry *d_plan = nullptr;
    uint32_t plan_cap = 0;
    size_t bytes_dir = 0, bytes_vals = 0, bytes_pool = 0, bytes_link = 0, bytes_live = 0, bytes_surv = 0; // sizes of the cached buffers
    SearchCtrl *d_ctrl = nullptr;
    SearchCtrl *h_ctrl = nullptr; // pinned
    uint32_t *d_trace = nullptr;  // backtrace output
    unsigned long long *d_live = nullptr;  // live parents of the round: (keyw + 1) arrays of live_cap u64
    uint64_t live_cap = 0;
    unsigned long long *d_surv = nullptr;  // local survivors of the round: pg_xrec records
    uint64_t surv_cap = 0;
    unsigned long long *d_host_counts = nullptr; // record counts the host passes to insert launches
    unsigned long long h_host_counts[64] = {0};
    pg_search_config cfg;
    int64_t batch_target = 0;
    int f0 = 0, f_range = 0, ub = 0;
    int goal_limit = 0;      // goals with g >= this are dropped (the all-advance cost + 1); weighted: every successor
    long long inc = LLONG_MAX; // the incumbent's cost U when the search began (LLONG_MAX: none)
    // multi-partition outboxes
    char *d_outbox = nullptr;
    unsigned long long *d_outbox_count = nullptr;
    unsigned long long *h_outbox_count = nullptr;
    uint64_t outbox_cap = 0; // records per destination
    void *peer_inbox[16] = {nullptr};
    unsigned long long *peer_counts[16] = {nullptr}; // P2P mode: every partition's uint64[nbuf][n_parts] "records from source s"
    int p2p_nbuf = 1, p2p_buf = 0;                   // double-buffered inboxes: one cross-GPU barrier per round is enough
    bool stamped = false;                            // counts carry the exchange round: receivers wait for them on the device, no barrier
    long long xround = 0;                            // exchange rounds completed
    bool p2p = false;
    bool forward = false;      // P2P parent forwarding (pg_search_config.reserved == 2)
    bool merge_expand = false; // forwarding: own and forwarded parents expanded by ONE launch after the barrier
    size_t region_bytes = 0;   // bytes one source may write into one inbox (per buffer)
    int xrec = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // optional per-launch timing: event triples (before select, between, after expand), harvested at every sync
    bool profile = false;
    std::vector<cudaEvent_t> prof_ev;
    size_t prof_used = 0;
    double expand_ms = 0, select_ms = 0, claim_ms = 0, insert_ms = 0, inbox_ms = 0;
    std::vector<cudaEvent_t> prof_ev2; // pairs around the inbox inserts
    size_t prof_used2 = 0;
    double kernel_ms = 0;
    int64_t rounds = 0;
    bool active = false;
    bool stepwise = true;    // begun by pg_search_begin (false: by pg_search, which has finished with it)
    // pg_run_rounds: a group of rounds captured once as a CUDA graph (every round is the same launches with the same
    // arguments; all per-round state lives in the device control block) and replayed
    GraphExec rounds_exec;
    int rounds_group = 0, rounds_flimit = 0;
    cudaStream_t rounds_stream = nullptr;
    bool rounds_no_graph = false; // a capture failed: this search runs its rounds as plain launches
};

struct pg_ctx {
    int device = 0;
    int n = 0, npairs = 0;
    int len[PG_MAX_SEQ] = {0};
    std::vector<std::string> seqs;
    std::vector<PairGeom> pairs;
    std::vector<int32_t> cost; // host copy of the 90 x 90 cost table (re-scoring of weighted-search alignments)
    DevProblem dp;
    uint8_t *d_seq = nullptr;
    int32_t *d_cost = nullptr;
    void *d_tables = nullptr;
    size_t table_cells = 0;
    bool tables_built = false;
    bool cost_u8 = false;      // every entry of the cost table is in 0..255 (the linear-gap DP kernel packs them in bytes)
    int n_alpha = 0;           // distinct residues over all sequences
    int sm_count = PG_SM_COUNT_B200;
    cudaStream_t stream = nullptr;       // stream all launches go to (own_stream unless pg_ctx_set_stream)
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream2 = nullptr;
    // staging for the host-pointer entry points
    void *d_stage[2] = {nullptr, nullptr};
    size_t stage_bytes[2] = {0, 0};
    SearchState *search = nullptr;
    // weighted search (pg_search_set_weight): f_w = g + h_w, h_w = sum of floor(wnum * term / 2^wsh); (1, 0) = exact A*
    int wnum = 1, wsh = 0;
    bool lb_valid = false;  // lower_bound holds the certified bound of the last pg_search / pg_multi_search
    int32_t lower_bound = 0;
    // incumbent (pg_search_set_incumbent): a known alignment and its cost U; every later search keeps only what can beat
    // U.  inc_cost < 0: none
    std::vector<std::string> inc_rows;
    long long inc_cost = -1;
    // resident CTAs per SM of the kernels that opt in to > 48 KB of dynamic shared memory; 0 = attribute not set yet on
    // this context's device (N and the key width are fixed per context, so one slot per kernel / mode is enough)
    int occ_expand_batch = 0;
    int occ_expand_probe[4] = {0, 0, 0, 0}; // per mode; [3] = mode 2 without per-successor owner arithmetic
    std::string err;
};

int pg_fail(pg_ctx *ctx, int code, const std::string &msg);
#define PG_CUDA(ctx, expr)                                                                                      \
    do {                                                                                                        \
        cudaError_t e__ = (expr);                                                                               \
        if (e__ != cudaSuccess)                                                                                 \
            return pg_fail(ctx, PG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));              \
    } while (0)

int pg_stage(pg_ctx *ctx, int which, size_t bytes, void **out);

// kernels' host launchers
int pg_launch_pair_dp(pg_ctx *ctx, float *kernel_ms);
int pg_launch_expand(pg_ctx *ctx, const void *d_parents, int64_t k, int vec_size, void *d_out, int32_t *d_counts,
                     cudaStream_t st);
int pg_launch_calc_h(pg_ctx *ctx, const uint16_t *d_coords, int64_t n, int32_t *d_out, cudaStream_t st);
int pg_launch_owner(pg_ctx *ctx, const uint16_t *d_coords, int64_t n, int size, uint32_t *d_out, cudaStream_t st);
void pg_search_free(pg_ctx *ctx);

// ---- the search internals the host drivers (pg_drivers.cu) build on (pg_search.cu) ------------------------------------
int sync_ctrl(pg_ctx *ctx); // control block to the host after a stream synchronise; a device-reported error as PG_ERR_*
void fill_counters(const SearchState *s, pg_result *r);
// Open / closed census of this partition's table and the min of g + h over its open entries (LLONG_MAX if none).
int pg_census(pg_ctx *ctx, int64_t *open_size, int64_t *closed_size, long long *open_lb);
// The parent chain from the goal to the origin: move masks origin-first, and the g stored at the goal entry.
int pg_backtrace(pg_ctx *ctx, std::vector<uint32_t> &masks, int *goal_g);
// Capture what `enqueue` launches on ctx->stream (thread-local mode) and instantiate it as *exec.  The captured rounds
// have not run, so the search's round count is restored.  A capture or instantiation the driver refuses leaves *exec
// empty and returns PG_OK; an error of `enqueue` is returned as it is.
int pg_capture(pg_ctx *ctx, const std::function<int()> &enqueue, GraphExec *exec);
// n rounds of a single-partition search.  allow_graph: whole groups of `group` rounds replay a CUDA graph, captured on
// first use and again when f_limit, the stream or the group size changes; after a failed capture the search does not try
// again.  The other rounds run as plain launches.
int pg_run_rounds(pg_ctx *ctx, int n, int f_limit, int group, bool allow_graph);
// g of the alignment spelled by `masks` (origin first) under the context's cost model (Node.cpp:129-152).
long long pg_path_cost(const pg_ctx *ctx, const std::vector<uint32_t> &masks);

// ---- device helpers ------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ int pg_pair_index(int n, int x, int y) // x < y, (i<j) order of HeuristicHPair.cpp:54-61
{
    return x * n - x * (x + 1) / 2 + (y - x - 1);
}

__device__ __forceinline__ int pg_table_cell(const DevProblem &p, int pair, int i, int j)
{
    size_t idx = (size_t)i * p.cols[pair] + j;
    if (p.cell16) return (int)__ldg(reinterpret_cast<const uint16_t *>(p.table[pair]) + idx);
    return __ldg(reinterpret_cast<const int32_t *>(p.table[pair]) + idx);
}

// Coord<N>::get_id (CoordHash.cpp:190-245) in closed form (SURVEY F5): the
// reference's z_order_hash writes floor(log2(size)) + shift%N + 2 Morton bits
// starting at coordinate bit shift/N, drops shift%N of them and takes % size.
// Bit m of the kept word is Morton bit (shift + m): coordinate (shift+m) % nd,
// bit (shift+m) / nd.  PZORDER is the same over coordinates 0 and 1 only.
__device__ __forceinline__ uint32_t pg_owner_of(const uint16_t *c, int n, int hash_type, int shift, int size, int log2size)
{
    if (hash_type == PG_HASH_FSUM) {
        unsigned s = 0;
        for (int i = 0; i < n; i++) s += c[i];
        return (s >> shift) % (unsigned)size;
    }
    if (hash_type == PG_HASH_PSUM) return ((unsigned)(c[0] + c[1]) >> shift) % (unsigned)size;
    int nd = hash_type == PG_HASH_PZORDER ? 2 : n;
    int nb = log2size + 2;
    unsigned w = 0;
    for (int m = 0; m < nb; m++) {
        int q = shift + m;
        int bit = q / nd;
        unsigned v = bit < 16 ? ((unsigned)c[q % nd] >> bit) & 1u : 0u;
        w |= v << m;
    }
    return w % (unsigned)size;
}
#endif
