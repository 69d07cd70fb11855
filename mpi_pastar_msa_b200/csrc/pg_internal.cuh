// Internal declarations shared by the CUDA translation units of libpastar_gpu.
// sm_100a only; no other architecture is built and there is no CPU path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

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

struct SearchState;
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
