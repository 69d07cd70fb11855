// Kernels of the layered (breadth-first heuristic) search, and the host code that runs one level pass over them.  The
// schedule of passes and the divide-and-conquer reconstruction are in pg_drivers.cu (pg_search_layered).
//
// Every move advances the level sum(pos) by 1 .. N, so the lattice is swept level by level in topological order: when
// level d is complete (levels d - N .. d - 1 expanded) its table is compacted into a list and expanded in one launch, and
// its successors go into the tables of levels d + 1 .. d + N.  A node is expanded once, with its final g; there is no
// open list and no closed list.  Relay mode holds a ring of N + 1 level tables; retain mode keeps every level of the box.
//
// Level table: open addressing over packed keys (KEYW=1 {key + 1}, KEYW=2 {lo, hi | 1 << 63}; 0 = free) with one u64
// value per slot, g << 32 | low, merged with atomicMin so that the smallest g wins (and among equal g the smallest low)
// whatever the order of the threads.  low is the parent move in retain mode; in relay mode it is the move into the node
// when that move crosses the middle level (low < RELAY_BASE) and RELAY_BASE + the relay's id otherwise.  Each claimed slot
// is also appended to the table's claim list, so compaction and clearing cost the level's width, not the table's size.
//
// A pass is the same three launches per level (compact, expand, advance): the level index and every counter live in the
// device control block, so a group of levels is captured once as a CUDA graph and replayed.
//
// Beam mode (width W > 0, pg_search_beam) is a relay-mode pass over the whole lattice with no crossing level: compaction
// writes the level's candidates to a staging list, and a cut between compaction and expansion keeps the W least by
// (f, packed key).  The cut is a radix select decided on the device (score, one launch per 8-bit digit of f - f_min and of
// the key, keep), so the launches of a level stay the same and replay as a graph.  Each kept node is appended to the
// retained array as {key, g << 32 | parent's retained index}, and its low in the expand list is its own retained index,
// so every successor carries its parent's index and the alignment is traced back from the goal's.
#include <algorithm>
#include <climits>
#include <cstring>
#include <vector>

#include "pg_expand_core.cuh"
#include "pg_key.cuh"

namespace {

constexpr int LAY_THREADS = 256;
constexpr int LAY_NB = PG_LAYERED_BINS;
constexpr uint32_t RELAY_BASE = 1u << 16;    // values of low below this are crossing moves (masks < 2^16)
constexpr unsigned long long VAL_EMPTY = ~0ull;
constexpr int LAY_GROUP = 16;                // levels per captured graph
constexpr int LAY_SYNC = 64;                 // levels between host checks (capacity, a dead pass, the budget)
constexpr unsigned LAY_MAX_PROBE = 4096;     // a longer probe sequence counts as a full table (the load is at most 1/2)

struct LayCtrl {
    int32_t d;           // the level compacted and expanded next
    int32_t error;       // 1: a level table is full
    int32_t dead;        // 1: nothing is left ahead of d: the pass cannot reach t
    int32_t fmin, fmax;  // over the successors that failed the bound only
    uint32_t list_n;     // nodes in the compacted list of level d
    uint32_t relay_n;    // relay entries saved
    uint32_t pad;
    unsigned long long expansions, generated, inserted, levels, max_level, max_held;
    // beam mode: the cut of level d
    uint32_t cand_n;             // candidates of level d before the cut
    uint32_t sel_all;            // 1: cand_n <= width, every candidate is kept
    uint32_t sel_done;           // 1: the kept set is decided
    uint32_t sel_k;              // candidates still to take from the tie class of the prefix
    uint32_t blocks_done;        // last-block handshake of the score and select kernels
    uint32_t keep_n;             // kept entries written so far
    int32_t lvl_fmin, lvl_fmax;  // f range of level d (score kernel accumulators)
    int32_t sel_f0;              // level d's least f: the select orders by the unsigned f - sel_f0, then the key
    uint32_t sel_fp, sel_fm;     // decided bits of f - sel_f0: prefix and mask
    int32_t drop_fmin;           // least f of the candidates the cut dropped
    unsigned long long sel_kp[2], sel_km[2]; // decided bits of the packed key (lo, hi word)
    unsigned long long ret_base, ret_n;      // first retained index of level d; retained entries so far
    unsigned long long dropped, max_cand;
};

struct DevLay {
    unsigned long long *keys;   // tables x S x KEYW
    unsigned long long *vals;   // tables x S
    uint32_t *claims;           // tables x L: the claimed slots of each table, in claim order
    uint32_t *counts;           // per table: claims so far
    unsigned long long smask;   // S - 1
    int lg_s;
    uint32_t L;                 // coordinates one level may hold
    int nt;                     // tables in use: N + 1 (relay ring) or lt - ls + 1 (retain)
    int retain;
    int n, kb;
    unsigned long long *list_key;  // KEYW x L, word-major
    unsigned long long *list_val;
    unsigned long long *relay_key; // KEYW x relay_cap, word-major
    unsigned long long *relay_val; // g << 32 | crossing move
    uint32_t relay_cap;
    int s[PG_MAX_SEQ], t[PG_MAX_SEQ];
    int ls, lt, mid;
    int U, strict;
    int hist_w;
    unsigned long long *hist;
    LayCtrl *ctrl;
    // beam mode
    uint32_t width;                // 0: no cut
    int kd;                        // 8-bit digits of the packed key: ceil(n kb / 8)
    unsigned long long *cand_key;  // KEYW x L, word-major: the level before the cut
    unsigned long long *cand_val;
    int32_t *cand_f;               // f of each candidate
    uint32_t *sel_hist;            // 256 bins of the select pass
    unsigned long long *ret_key;   // KEYW x ret_cap, word-major
    unsigned long long *ret_val;   // g << 32 | the parent's retained index (~0: the origin)
    unsigned long long ret_cap;
};

__device__ __forceinline__ int lay_table(const DevLay &d, int level) { return d.retain ? level - d.ls : level % d.nt; }

template <int KEYW>
__device__ __forceinline__ unsigned long long *lay_key_ptr(const DevLay &d, int ti, unsigned long long slot)
{
    return d.keys + (((unsigned long long)ti << d.lg_s) + slot) * KEYW;
}

template <int KEYW>
__device__ __forceinline__ bool lay_key_is(const unsigned long long h0, const unsigned long long h1, const Key<KEYW> &k)
{
    if constexpr (KEYW == 1)
        return h0 == k.lo + 1;
    else
        return h0 == k.lo && h1 == (k.hi | (1ull << 63));
}

template <int KEYW>
__device__ __forceinline__ Key<KEYW> lay_key_decode(const unsigned long long h0, const unsigned long long h1)
{
    Key<KEYW> k;
    if constexpr (KEYW == 1) {
        k.lo = h0 - 1;
    } else {
        k.lo = h0;
        k.hi = h1 & ~(1ull << 63);
    }
    return k;
}

// Slot of `k` in table ti, claimed when absent and `claim` (fresh = true then); ~0 when absent, or when no slot was found
// within LAY_MAX_PROBE probes (the table is full).
template <int KEYW>
__device__ __forceinline__ unsigned long long lay_find(const DevLay &d, int ti, const Key<KEYW> &k, bool claim, bool &fresh)
{
    fresh = false;
    unsigned long long slot = d.lg_s ? (unsigned long long)((unsigned)k.hash() >> (32 - d.lg_s)) : 0ull;
    for (unsigned probe = 0; probe < LAY_MAX_PROBE && probe <= d.smask; probe++, slot = (slot + 1) & d.smask) {
        unsigned long long *e = lay_key_ptr<KEYW>(d, ti, slot);
        unsigned long long h0, h1 = 0;
        if constexpr (KEYW == 1)
            h0 = ld_cg_u64(e);
        else
            ld_cg_v2(e, h0, h1);
        if (lay_key_is<KEYW>(h0, h1, k)) return slot;
        if (h0 != 0 || h1 != 0) continue;
        if (!claim) return ~0ull;
        if constexpr (KEYW == 1) {
            const unsigned long long prev = atomicCAS(e, 0ull, k.lo + 1);
            if (prev == 0) fresh = true;
            if (prev == 0 || prev == k.lo + 1) return slot;
        } else {
            unsigned long long p0, p1;
            cas128(e, k.lo, k.hi | (1ull << 63), p0, p1);
            if (p0 == 0 && p1 == 0) fresh = true;
            if (fresh || lay_key_is<KEYW>(p0, p1, k)) return slot;
        }
    }
    return ~0ull;
}

// Enter `k` into the table of level `level` with value v (atomicMin); true when it claimed a new slot.
template <int KEYW>
__device__ __forceinline__ bool lay_insert(const DevLay &d, int level, const Key<KEYW> &k, unsigned long long v)
{
    if (*(volatile int32_t *)&d.ctrl->error) return false; // the pass fails with PG_ERR_CAPACITY: do not fill the table
    const int ti = lay_table(d, level);
    bool fresh;
    const unsigned long long slot = lay_find<KEYW>(d, ti, k, true, fresh);
    if (slot == ~0ull) {
        d.ctrl->error = 1;
        return false;
    }
    if (fresh) {
        const uint32_t at = atomicAdd(d.counts + ti, 1u);
        if (at >= d.L)
            d.ctrl->error = 1;
        else
            d.claims[(size_t)ti * d.L + at] = (uint32_t)slot;
    }
    atomicMin(d.vals + ((unsigned long long)ti << d.lg_s) + slot, v);
    return fresh;
}

template <int KEYW>
__device__ __forceinline__ Key<KEYW> lay_pos_key(const DevLay &d, const int *pos)
{
    Key<KEYW> k = Key<KEYW>::zero();
    for (int i = 0; i < d.n; i++) k.add_val((unsigned)pos[i], i * d.kb);
    return k;
}

// s enters its level's table with g0 and low0; the control block starts the pass at level(s)
template <int KEYW>
__global__ void layered_seed_kernel(const __grid_constant__ DevLay d, int g0, uint32_t low0)
{
    LayCtrl *c = d.ctrl;
    c->d = d.ls;
    c->fmin = c->lvl_fmin = c->drop_fmin = INT_MAX;
    c->fmax = c->lvl_fmax = INT_MIN;
    const Key<KEYW> k = lay_pos_key<KEYW>(d, d.s);
    lay_insert<KEYW>(d, d.ls, k, ((unsigned long long)(unsigned)g0 << 32) | low0);
    c->inserted = 1;
}

// Level d's table as a {key, g << 32 | low} list.  Relay mode clears every slot it reads (the table serves level
// d + N + 1 next) and gives each node of the levels mid + 1 .. mid + N that was entered by a crossing move a relay id.
template <int KEYW>
__global__ void __launch_bounds__(LAY_THREADS) layered_compact_kernel(const __grid_constant__ DevLay d)
{
    LayCtrl *c = d.ctrl;
    if (c->dead || c->error) return;
    const int lv = c->d;
    const int ti = lay_table(d, lv);
    const uint32_t n = min(d.counts[ti], d.L);
    const bool band = !d.retain && lv > d.mid && lv <= d.mid + d.n;
    if (blockIdx.x == 0 && threadIdx.x == 0) c->list_n = n;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long slot = d.claims[(size_t)ti * d.L + i];
        unsigned long long *e = lay_key_ptr<KEYW>(d, ti, slot);
        unsigned long long *vp = d.vals + ((unsigned long long)ti << d.lg_s) + slot;
        const unsigned long long h0 = e[0], h1 = KEYW == 2 ? e[1] : 0ull;
        unsigned long long v = *vp;
        if (!d.retain) {
            e[0] = 0;
            if constexpr (KEYW == 2) e[1] = 0;
            *vp = VAL_EMPTY;
        }
        const Key<KEYW> k = lay_key_decode<KEYW>(h0, h1);
        if (band && (uint32_t)v < RELAY_BASE) {
            const uint32_t id = atomicAdd(&c->relay_n, 1u); // relay_cap = N x L: never short
            d.relay_key[id] = k.lo;
            if constexpr (KEYW == 2) d.relay_key[d.relay_cap + id] = k.hi;
            d.relay_val[id] = v;
            v = (v & 0xffffffff00000000ull) | (RELAY_BASE + id);
        }
        d.list_key[i] = k.lo;
        if constexpr (KEYW == 2) d.list_key[d.L + i] = k.hi;
        d.list_val[i] = v;
    }
}

template <int N, int KEYW>
struct LayerSink {
    const DevLay &d;
    int level;      // the parent's level
    uint32_t low;   // the parent's low
    int *s_hist;
    unsigned gen, ins;
    int fmin, fmax;
    __device__ __forceinline__ void operator()(int mask, int, const int (&posn)[N], int gnew, int hnew)
    {
        gen++;
        bool in = true;
#pragma unroll
        for (int i = 0; i < N; i++) in &= posn[i] <= d.t[i];
        if (!in) return;
        const int f = gnew + hnew;
        if (d.strict ? f >= d.U : f > d.U) {
            fmin = min(fmin, f);
            fmax = max(fmax, f);
            atomicAdd(s_hist + min((unsigned)(f - d.U) / (unsigned)d.hist_w, (unsigned)(LAY_NB - 1)), 1);
            return;
        }
        Key<KEYW> k = Key<KEYW>::zero();
#pragma unroll
        for (int i = 0; i < N; i++) k.add_val((unsigned)posn[i], i * d.kb);
        const int lv2 = level + __popc(mask);
        const uint32_t lo = d.retain ? (uint32_t)mask : (level <= d.mid && lv2 > d.mid ? (uint32_t)mask : low);
        ins += lay_insert<KEYW>(d, lv2, k, ((unsigned long long)(unsigned)gnew << 32) | lo);
    }
};

// Expand level d's list: a group of ExpCfg<N>::LP lanes per parent (pg_expand_parent), the box and bound tests and the
// level-table insert in the sink; f_min / f_max and the histogram of the pruned f go through shared memory.
template <int N, int KEYW>
__global__ void __launch_bounds__(LAY_THREADS) layered_expand_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevLay d)
{
    using C = ExpCfg<N>;
    constexpr int GROUPS = LAY_THREADS / C::LP;
    LayCtrl *c = d.ctrl;
    if (c->dead || c->error) return;
    const uint32_t n = c->list_n;
    if ((unsigned long long)blockIdx.x * GROUPS >= n) return; // whole CTA
    const int lv = c->d;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PairMeta *meta = reinterpret_cast<PairMeta *>(smem_raw);
    int *s_hist = reinterpret_cast<int *>(smem_raw + ((sizeof(PairMeta) + 15) & ~size_t(15)));
    int *s_red = s_hist + LAY_NB; // fmin, fmax, generated, inserted
    int *s_groups = s_red + 4;
    pg_load_pair_meta(p, meta);
    for (int i = threadIdx.x; i < LAY_NB; i += blockDim.x) s_hist[i] = 0;
    if (threadIdx.x == 0) {
        s_red[0] = INT_MAX;
        s_red[1] = INT_MIN;
        s_red[2] = s_red[3] = 0;
    }
    __syncthreads();

    const int grp = threadIdx.x / C::LP, sub = threadIdx.x % C::LP;
    const int lane = threadIdx.x & 31;
    const unsigned gmask = C::LP == 32 ? 0xffffffffu : (((1u << C::LP) - 1u) << (lane & ~(C::LP - 1)));
    int *s_grp = s_groups + grp * C::GROUP_INTS;
    const unsigned fmask = (1u << d.kb) - 1u;
    LayerSink<N, KEYW> sink{d, lv, 0u, s_hist, 0u, 0u, INT_MAX, INT_MIN};
    for (unsigned long long base = (unsigned long long)blockIdx.x * GROUPS; base < n; base += (unsigned long long)gridDim.x * GROUPS) {
        const unsigned long long pi = base + grp;
        if (pi >= n) continue; // whole group
        Key<KEYW> k;
        k.lo = d.list_key[pi];
        if constexpr (KEYW == 2) k.hi = d.list_key[d.L + pi];
        const unsigned long long v = d.list_val[pi];
        int pos[N];
#pragma unroll
        for (int i = 0; i < N; i++) pos[i] = (int)k.field(i * d.kb, fmask);
        sink.low = (uint32_t)v;
        // gap_open == gap_ext (pg_search_layered refuses other models): the incoming move does not change a cost
        pg_expand_parent<N>(p, meta, s_grp, pos, (int)(v >> 32), (1 << N) - 1, sub, gmask, sink);
    }
    if (sink.fmin != INT_MAX) atomicMin(s_red + 0, sink.fmin);
    if (sink.fmax != INT_MIN) atomicMax(s_red + 1, sink.fmax);
    atomicAdd(s_red + 2, (int)sink.gen);
    atomicAdd(s_red + 3, (int)sink.ins);
    __syncthreads();
    for (int i = threadIdx.x; i < LAY_NB; i += blockDim.x)
        if (s_hist[i]) atomicAdd(d.hist + i, (unsigned long long)s_hist[i]);
    if (threadIdx.x == 0) {
        if (s_red[0] != INT_MAX) atomicMin(&c->fmin, s_red[0]);
        if (s_red[1] != INT_MIN) atomicMax(&c->fmax, s_red[1]);
        atomicAdd(&c->generated, (unsigned long long)(unsigned)s_red[2]);
        atomicAdd(&c->inserted, (unsigned long long)(unsigned)s_red[3]);
    }
}

// After level d: counters, the coordinates held, the ring slot of level d freed, d + 1, and whether anything is left.
__global__ void layered_advance_kernel(const __grid_constant__ DevLay d)
{
    LayCtrl *c = d.ctrl;
    if (c->dead || c->error) return;
    const int lv = c->d;
    c->expansions += c->list_n;
    c->levels++;
    c->max_level = max(c->max_level, (unsigned long long)c->list_n);
    unsigned long long held = 0, ahead = 0;
    if (d.retain) {
        held = c->inserted;
        for (int l = lv + 1; l <= min(lv + d.n, d.lt); l++) ahead += d.counts[lay_table(d, l)];
    } else {
        for (int i = 0; i < d.nt; i++) held += d.counts[i];
        d.counts[lay_table(d, lv)] = 0;
        for (int i = 0; i < d.nt; i++) ahead += d.counts[i];
    }
    c->max_held = max(c->max_held, held);
    c->list_n = 0;
    c->d = lv + 1;
    if (ahead == 0) c->dead = 1;
}

// Every claimed slot of the first nt tables back to empty (the slots a pass left behind: its last level, or the levels
// after it stopped, or all of a retain pass)
template <int KEYW>
__global__ void __launch_bounds__(LAY_THREADS) layered_clear_kernel(const __grid_constant__ DevLay d)
{
    const int ti = blockIdx.y;
    const uint32_t n = min(d.counts[ti], d.L);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long slot = d.claims[(size_t)ti * d.L + i];
        unsigned long long *e = lay_key_ptr<KEYW>(d, ti, slot);
        e[0] = 0;
        if constexpr (KEYW == 2) e[1] = 0;
        d.vals[((unsigned long long)ti << d.lg_s) + slot] = VAL_EMPTY;
    }
}

// Retain mode: the parent masks from t back to s.  out[0] = moves (or ~0 when the chain breaks), out[1] = g(t),
// out[2 ..] = the masks, t first.
template <int KEYW>
__global__ void layered_trace_kernel(const __grid_constant__ DevLay d, uint32_t *out, int max_moves)
{
    int cur[PG_MAX_SEQ];
    int lv = 0;
    for (int i = 0; i < d.n; i++) {
        cur[i] = d.t[i];
        lv += cur[i];
    }
    int k = 0;
    for (;;) {
        bool fresh;
        const Key<KEYW> key = lay_pos_key<KEYW>(d, cur);
        const int ti = lay_table(d, lv);
        const unsigned long long slot = lay_find<KEYW>(d, ti, key, false, fresh);
        if (slot == ~0ull) break;
        const unsigned long long v = d.vals[((unsigned long long)ti << d.lg_s) + slot];
        if (k == 0) out[1] = (uint32_t)(v >> 32);
        if (lv == d.ls) { // s: the only node of its level in the box
            out[0] = (uint32_t)k;
            return;
        }
        const uint32_t m = (uint32_t)v;
        if (k >= max_moves || m == 0 || m >= (1u << d.n)) break;
        out[2 + k++] = m;
        for (int i = 0; i < d.n; i++) cur[i] -= (m >> i) & 1;
        lv -= __popc(m);
        if (lv < d.ls) break;
    }
    out[0] = ~0u;
}

// ---- beam mode: the cut of level d ----------------------------------------------------------------------------------

template <int KEYW>
__device__ __forceinline__ Key<KEYW> beam_cand_key(const DevLay &d, uint32_t i)
{
    Key<KEYW> k;
    k.lo = d.cand_key[i];
    if constexpr (KEYW == 2) k.hi = d.cand_key[d.L + i];
    return k;
}

// true in every thread of the last block of the grid to get here; the other blocks' atomics are then visible
__device__ __forceinline__ bool beam_last_block(LayCtrl *c)
{
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(&c->blocks_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last) __threadfence();
    return last;
}

// f = g + h of every candidate (h as pg_calculate_h: the sum over pairs of the table cell x w); the last block reads the
// level's f range and starts the select: every candidate is kept when they number at most W, else the bits of f - f_min
// above the range's highest set bit are decided (all zero) and the W least by (f, key) remain to be found.
template <int N, int KEYW>
__global__ void __launch_bounds__(LAY_THREADS) beam_score_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevLay d)
{
    LayCtrl *c = d.ctrl;
    if (c->dead || c->error) return;
    const uint32_t n = c->list_n;
    const unsigned fmask = (1u << d.kb) - 1u;
    int lo = INT_MAX, hi = INT_MIN;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const Key<KEYW> k = beam_cand_key<KEYW>(d, i);
        int pos[N];
#pragma unroll
        for (int x = 0; x < N; x++) pos[x] = (int)k.field(x * d.kb, fmask);
        int h = 0;
#pragma unroll
        for (int x = 0; x < N; x++)
#pragma unroll
            for (int y = x + 1; y < N; y++) {
                const int pr = x * N - x * (x + 1) / 2 + (y - x - 1);
                h += pg_table_cell(p, pr, pos[x], pos[y]) * p.w[pr];
            }
        const int f = (int)(d.cand_val[i] >> 32) + h;
        d.cand_f[i] = f;
        lo = min(lo, f);
        hi = max(hi, f);
    }
    for (int o = 16; o; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0 && lo != INT_MAX) {
        atomicMin(&c->lvl_fmin, lo);
        atomicMax(&c->lvl_fmax, hi);
    }
    if (!beam_last_block(c) || threadIdx.x != 0) return;
    volatile LayCtrl *vc = c;
    const int f0 = vc->lvl_fmin, f1 = vc->lvl_fmax;
    const uint32_t k = min(n, d.width);
    c->lvl_fmin = INT_MAX;
    c->lvl_fmax = INT_MIN;
    c->blocks_done = 0;
    c->cand_n = n;
    c->max_cand = max(c->max_cand, (unsigned long long)n);
    c->ret_base = c->ret_n;
    c->ret_n += k;
    if (c->ret_n > d.ret_cap) c->error = 1; // the host sized the array for every level: not reached
    c->dropped += n - k;
    c->keep_n = 0;
    c->sel_all = c->sel_done = n <= d.width;
    c->sel_k = k;
    c->sel_f0 = f0;
    const int z = __clz((int)((unsigned)f1 - (unsigned)f0));
    c->sel_fp = 0;
    c->sel_fm = z == 0 ? 0u : ~0u << (32 - z);
    c->sel_kp[0] = c->sel_kp[1] = c->sel_km[0] = c->sel_km[1] = 0;
}

// The decided bits of the select, in registers: a candidate's (f - f0, key) under the masks against the prefix
struct BeamSel {
    unsigned f0, fp, fm;
    unsigned long long kp[2], km[2];
    __device__ __forceinline__ explicit BeamSel(const LayCtrl *c)
        : f0((unsigned)c->sel_f0), fp(c->sel_fp), fm(c->sel_fm), kp{c->sel_kp[0], c->sel_kp[1]}, km{c->sel_km[0], c->sel_km[1]}
    {
    }
    // -1, 0, 1: below, in, above the tie class of the prefix
    template <int KEYW>
    __device__ __forceinline__ int cmp(int f, const Key<KEYW> &k) const
    {
        const unsigned a = ((unsigned)f - f0) & fm;
        if (a != fp) return a < fp ? -1 : 1;
        if constexpr (KEYW == 2) {
            const unsigned long long h = k.hi & km[1];
            if (h != kp[1]) return h < kp[1] ? -1 : 1;
        }
        const unsigned long long l = k.lo & km[0];
        return l == kp[0] ? 0 : (l < kp[0] ? -1 : 1);
    }
};

// One radix-select pass: digit 0 .. 3 are the bytes of f - f_min from the top, digit 4 + j byte kd - 1 - j of the packed
// key.  The candidates in the tie class are counted by the digit's value; the last block finds the bin that holds the
// sel_k-th of them and adds it to the prefix.  When that bin holds exactly the candidates still wanted, the cut is decided.
template <int KEYW>
__global__ void __launch_bounds__(LAY_THREADS) beam_select_kernel(const __grid_constant__ DevLay d, int digit)
{
    LayCtrl *c = d.ctrl;
    if (c->dead || c->error || c->sel_done) return;
    const bool fd = digit < 4;
    const int sh = fd ? 24 - 8 * digit : 8 * (d.kd - 1 - (digit - 4));
    if (fd && ((c->sel_fm >> sh) & 0xffu) == 0xffu) return; // decided by the f range
    __shared__ uint32_t s_h[256];
    for (int b = threadIdx.x; b < 256; b += blockDim.x) s_h[b] = 0;
    __syncthreads();
    const uint32_t n = c->cand_n;
    const BeamSel sel(c);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int f = d.cand_f[i];
        const Key<KEYW> k = beam_cand_key<KEYW>(d, i);
        if (sel.cmp<KEYW>(f, k) != 0) continue;
        unsigned long long word = (unsigned)f - sel.f0;
        if (!fd) {
            word = k.lo;
            if constexpr (KEYW == 2)
                if (sh >= 64) word = k.hi;
        }
        const uint32_t v = (uint32_t)(word >> (sh & 63)) & 0xffu;
        atomicAdd(s_h + v, 1u);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < 256; b += blockDim.x)
        if (s_h[b]) atomicAdd(d.sel_hist + b, s_h[b]);
    if (!beam_last_block(c) || threadIdx.x != 0) return;
    volatile uint32_t *h = d.sel_hist;
    const uint32_t want = c->sel_k;
    uint32_t below = 0, b = 0;
    for (; b < 255 && below + h[b] < want; b++) below += h[b];
    const uint32_t rest = want - below;
    if (fd) {
        c->sel_fp |= b << sh;
        c->sel_fm |= 0xffu << sh;
    } else {
        c->sel_kp[sh >> 6] |= (unsigned long long)b << (sh & 63);
        c->sel_km[sh >> 6] |= 0xffull << (sh & 63);
    }
    c->sel_k = rest;
    if (h[b] == rest) c->sel_done = 1;
    for (int i = 0; i < 256; i++) h[i] = 0;
    c->blocks_done = 0;
}

// The kept candidates (all, or those whose decided bits are at most the prefix) to the expand list and the retained
// array; the least f of the dropped ones to drop_fmin.
template <int KEYW>
__global__ void __launch_bounds__(LAY_THREADS) beam_keep_kernel(const __grid_constant__ DevLay d)
{
    LayCtrl *c = d.ctrl;
    if (c->dead || c->error) return;
    const uint32_t n = c->cand_n;
    const bool all = c->sel_all;
    const BeamSel sel(c);
    const unsigned long long base = c->ret_base;
    const int lane = threadIdx.x & 31;
    int dmin = INT_MAX;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i0 = blockIdx.x * blockDim.x; i0 < n; i0 += stride) { // warp-uniform trip count
        const uint32_t i = i0 + threadIdx.x;
        bool keep = false;
        Key<KEYW> k = Key<KEYW>::zero();
        unsigned long long v = 0;
        if (i < n) {
            const int f = d.cand_f[i];
            k = beam_cand_key<KEYW>(d, i);
            v = d.cand_val[i];
            keep = all || sel.cmp<KEYW>(f, k) <= 0;
            if (!keep) dmin = min(dmin, f);
        }
        const unsigned ball = __ballot_sync(0xffffffffu, keep);
        uint32_t at = 0;
        if (lane == 0 && ball) at = atomicAdd(&c->keep_n, (uint32_t)__popc(ball));
        at = __shfl_sync(0xffffffffu, at, 0) + __popc(ball & ((1u << lane) - 1u));
        if (keep) {
            const unsigned long long r = base + at;
            d.list_key[at] = k.lo;
            d.ret_key[r] = k.lo;
            if constexpr (KEYW == 2) {
                d.list_key[d.L + at] = k.hi;
                d.ret_key[d.ret_cap + r] = k.hi;
            }
            d.list_val[at] = (v & 0xffffffff00000000ull) | (uint32_t)r;
            d.ret_val[r] = v;
        }
    }
    for (int o = 16; o; o >>= 1) dmin = min(dmin, __shfl_xor_sync(0xffffffffu, dmin, o));
    if (lane == 0 && dmin != INT_MAX) atomicMin(&c->drop_fmin, dmin);
    if (blockIdx.x == 0 && threadIdx.x == 0) c->list_n = min(n, d.width); // the expand kernel's count; n stays in cand_n
}

// The moves from the origin to t: from the retained entry `at` (t's parent) along the parent indices.  out[0] = moves
// (~0 when the chain breaks), out[1] unused, out[2 ..] = the masks, t first.
template <int KEYW>
__global__ void beam_trace_kernel(const __grid_constant__ DevLay d, uint32_t at, uint32_t *out, int max_moves)
{
    int cur[PG_MAX_SEQ];
    for (int i = 0; i < d.n; i++) cur[i] = d.t[i];
    const unsigned fmask = (1u << d.kb) - 1u;
    int k = 0;
    out[0] = ~0u;
    for (; at != ~0u; k++) {
        if (k >= max_moves || at >= d.ret_cap) return;
        Key<KEYW> key;
        key.lo = d.ret_key[at];
        if constexpr (KEYW == 2) key.hi = d.ret_key[d.ret_cap + at];
        uint32_t m = 0;
        for (int i = 0; i < d.n; i++) {
            const int q = (int)key.field(i * d.kb, fmask), step = cur[i] - q;
            if (step != 0 && step != 1) return;
            m |= (uint32_t)step << i;
            cur[i] = q;
        }
        if (m == 0) return;
        out[2 + k] = m;
        at = (uint32_t)d.ret_val[at];
    }
    for (int i = 0; i < d.n; i++)
        if (cur[i] != d.s[i]) return;
    out[0] = (uint32_t)k;
}

template <int N, int KEYW>
size_t expand_smem()
{
    using C = ExpCfg<N>;
    return ((sizeof(PairMeta) + 15) & ~size_t(15)) + sizeof(int) * ((size_t)LAY_NB + 4 + (size_t)(LAY_THREADS / C::LP) * C::GROUP_INTS);
}

template <int N, int KEYW>
int launch_level_expand(pg_ctx *ctx, const DevLay &d, int grid)
{
    layered_expand_kernel<N, KEYW><<<grid, LAY_THREADS, expand_smem<N, KEYW>(), ctx->stream>>>(ctx->dp, d);
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

template <int N, int KEYW>
int launch_beam_score(pg_ctx *ctx, const DevLay &d, int grid)
{
    beam_score_kernel<N, KEYW><<<grid, LAY_THREADS, 0, ctx->stream>>>(ctx->dp, d);
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

template <int N, int KEYW>
int expand_attr(pg_ctx *ctx, int *grid)
{
    const size_t smem = expand_smem<N, KEYW>();
    PG_CUDA(ctx, cudaFuncSetAttribute(layered_expand_kernel<N, KEYW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    PG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, layered_expand_kernel<N, KEYW>, LAY_THREADS, smem));
    *grid = ctx->sm_count * std::max(occ, 1);
    return PG_OK;
}

} // namespace

struct LayeredState {
    int keyw = 1, n = 0;
    int64_t L = 0;               // coordinates per level
    int lg_s = 0;
    int n_tables = 0;            // allocated: max(N + 1, retain levels)
    unsigned long long *keys = nullptr, *vals = nullptr, *list_key = nullptr, *list_val = nullptr, *relay_key = nullptr,
                       *relay_val = nullptr, *hist = nullptr;
    uint32_t *claims = nullptr, *counts = nullptr, *trace = nullptr;
    // beam mode: the candidates before the cut, the select's bins, the retained array and the trace's output
    unsigned long long *cand_key = nullptr, *cand_val = nullptr, *ret_key = nullptr, *ret_val = nullptr;
    int32_t *cand_f = nullptr;
    uint32_t *sel_hist = nullptr, *beam_trace = nullptr;
    int64_t ret_cap = 0;
    LayCtrl *d_ctrl = nullptr, *h_ctrl = nullptr;
    int64_t bytes = 0;
    int expand_grid = 0, compact_grid = 0;
    bool no_graph = false;
};

namespace {

int lay_alloc(pg_ctx *ctx, LayeredState *L, void **p, size_t bytes)
{
    PG_CUDA(ctx, cudaMalloc(p, bytes));
    L->bytes += (int64_t)bytes;
    return PG_OK;
}

int beam_score(pg_ctx *ctx, const DevLay &d, int grid)
{
    const int kw = ctx->n * ctx->dp.key_bits <= 63 ? 1 : 2;
    switch (ctx->n * 2 + kw - 1) {
#define CASE(X)                                                                                                   \
    case 2 * X:                                                                                                   \
        return launch_beam_score<X, 1>(ctx, d, grid);                                                             \
    case 2 * X + 1:                                                                                               \
        return launch_beam_score<X, 2>(ctx, d, grid);
        CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
    default:
        return pg_fail(ctx, PG_ERR_ARG, "pg_search_beam: unsupported number of sequences");
    }
}

int lay_expand(pg_ctx *ctx, const DevLay &d, int grid, bool attr_only, int *grid_out)
{
    const int kw = ctx->n * ctx->dp.key_bits <= 63 ? 1 : 2;
    switch (ctx->n * 2 + kw - 1) {
#define CASE(X)                                                                                                   \
    case 2 * X:                                                                                                   \
        return attr_only ? expand_attr<X, 1>(ctx, grid_out) : launch_level_expand<X, 1>(ctx, d, grid);            \
    case 2 * X + 1:                                                                                               \
        return attr_only ? expand_attr<X, 2>(ctx, grid_out) : launch_level_expand<X, 2>(ctx, d, grid);
        CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
    default:
        return pg_fail(ctx, PG_ERR_ARG, "pg_search_layered: unsupported number of sequences");
    }
}

DevLay make_dev(const pg_ctx *ctx, const LayeredState *L, const LayPassIn &in)
{
    DevLay d;
    memset(&d, 0, sizeof(d));
    d.keys = L->keys;
    d.vals = L->vals;
    d.claims = L->claims;
    d.counts = L->counts;
    d.lg_s = L->lg_s;
    d.smask = (1ull << L->lg_s) - 1;
    d.L = (uint32_t)L->L;
    d.n = ctx->n;
    d.kb = ctx->dp.key_bits;
    d.list_key = L->list_key;
    d.list_val = L->list_val;
    d.relay_key = L->relay_key;
    d.relay_val = L->relay_val;
    d.relay_cap = (uint32_t)(L->L * ctx->n);
    d.ls = d.lt = 0;
    for (int i = 0; i < ctx->n; i++) {
        d.s[i] = in.s[i];
        d.t[i] = in.t[i];
        d.ls += in.s[i];
        d.lt += in.t[i];
    }
    d.retain = in.retain;
    d.nt = in.retain ? d.lt - d.ls + 1 : ctx->n + 1;
    d.mid = in.mid;
    d.U = in.U;
    d.strict = in.strict;
    d.hist_w = std::max(1, in.hist_w);
    d.hist = L->hist;
    d.ctrl = L->d_ctrl;
    d.width = (uint32_t)std::min<int64_t>(in.width, UINT32_MAX);
    d.kd = (ctx->n * ctx->dp.key_bits + 7) / 8;
    d.cand_key = L->cand_key;
    d.cand_val = L->cand_val;
    d.cand_f = L->cand_f;
    d.sel_hist = L->sel_hist;
    d.ret_key = L->ret_key;
    d.ret_val = L->ret_val;
    d.ret_cap = (unsigned long long)L->ret_cap;
    return d;
}

// the view the compact kernel writes through: in beam mode the level goes to the candidate list, not the expand list
DevLay compact_view(const DevLay &d)
{
    DevLay c = d;
    if (d.width) {
        c.list_key = d.cand_key;
        c.list_val = d.cand_val;
    }
    return c;
}

int launch_compact(pg_ctx *ctx, const LayeredState *L, const DevLay &d, int grid)
{
    const DevLay c = compact_view(d);
    if (L->keyw == 1)
        layered_compact_kernel<1><<<grid, LAY_THREADS, 0, ctx->stream>>>(c);
    else
        layered_compact_kernel<2><<<grid, LAY_THREADS, 0, ctx->stream>>>(c);
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

// the cut of the compacted level: score, one select pass per digit (4 of f, kd of the key), keep
int launch_cut(pg_ctx *ctx, const LayeredState *L, const DevLay &d)
{
    int rc = beam_score(ctx, d, L->compact_grid);
    if (rc != PG_OK) return rc;
    for (int digit = 0; digit < 4 + d.kd; digit++) {
        if (L->keyw == 1)
            beam_select_kernel<1><<<L->compact_grid, LAY_THREADS, 0, ctx->stream>>>(d, digit);
        else
            beam_select_kernel<2><<<L->compact_grid, LAY_THREADS, 0, ctx->stream>>>(d, digit);
    }
    if (L->keyw == 1)
        beam_keep_kernel<1><<<L->compact_grid, LAY_THREADS, 0, ctx->stream>>>(d);
    else
        beam_keep_kernel<2><<<L->compact_grid, LAY_THREADS, 0, ctx->stream>>>(d);
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

int launch_level(pg_ctx *ctx, const LayeredState *L, const DevLay &d)
{
    int rc = launch_compact(ctx, L, d, L->compact_grid);
    if (rc == PG_OK && d.width) rc = launch_cut(ctx, L, d);
    if (rc != PG_OK) return rc;
    rc = lay_expand(ctx, d, L->expand_grid, false, nullptr);
    if (rc != PG_OK) return rc;
    layered_advance_kernel<<<1, 1, 0, ctx->stream>>>(d);
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

int read_ctrl(pg_ctx *ctx, LayeredState *L)
{
    PG_CUDA(ctx, cudaMemcpyAsync(L->h_ctrl, L->d_ctrl, sizeof(LayCtrl), cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PG_OK;
}

} // namespace

int pg_layered_open(pg_ctx *ctx, int64_t level_cap, int retain_levels, int64_t beam_retained, LayeredState **out)
{
    *out = nullptr;
    LayeredState *L = new LayeredState();
    L->n = ctx->n;
    L->keyw = ctx->n * ctx->dp.key_bits <= 63 ? 1 : 2;
    L->L = std::max<int64_t>(1, std::min<int64_t>(level_cap, 1LL << 30));
    L->lg_s = 1;
    while ((1LL << L->lg_s) < 2 * L->L) L->lg_s++; // load factor at most one half
    L->n_tables = std::max(ctx->n + 1, retain_levels);
    L->no_graph = getenv("PG_NO_GRAPH") != nullptr;
    L->ret_cap = beam_retained;
    *out = L;
    const size_t S = (size_t)1 << L->lg_s, T = (size_t)L->n_tables;
    int rc;
    if (beam_retained > 0) {
        int D = 0;
        for (int i = 0; i < ctx->n; i++) D += ctx->len[i];
        const size_t kw = (size_t)L->keyw, Lc = (size_t)L->L, R = (size_t)beam_retained;
        const size_t need = T * S * kw * 8 + T * S * 8 + T * Lc * 4 + T * 4 + 2 * (Lc * kw * 8 + Lc * 8) + Lc * 4 + 256 * 4 +
                            R * (kw * 8 + 8) + ((size_t)D + 2) * 4 + LAY_NB * 8 + ((size_t)T + 2) * 4 + sizeof(LayCtrl);
        size_t free_b = 0, total_b = 0;
        PG_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
        if (need > free_b)
            return pg_fail(ctx, PG_ERR_CAPACITY, "pg_search_beam: " + std::to_string(need) + " bytes of level tables and retained array, " +
                                                     std::to_string(free_b) + " free on the device");
        if ((rc = lay_alloc(ctx, L, (void **)&L->cand_key, Lc * kw * 8)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->cand_val, Lc * 8)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->cand_f, Lc * 4)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->sel_hist, 256 * 4)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->ret_key, R * kw * 8)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->ret_val, R * 8)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->beam_trace, ((size_t)D + 2) * 4)) != PG_OK) return rc;
        PG_CUDA(ctx, cudaMemsetAsync(L->sel_hist, 0, 256 * 4, ctx->stream));
    }
    if ((rc = lay_alloc(ctx, L, (void **)&L->keys, T * S * L->keyw * 8)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->vals, T * S * 8)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->claims, T * L->L * 4)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->counts, T * 4)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->list_key, (size_t)L->L * L->keyw * 8)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->list_val, (size_t)L->L * 8)) != PG_OK) return rc;
    if (beam_retained == 0) { // beam passes have no relays
        if ((rc = lay_alloc(ctx, L, (void **)&L->relay_key, (size_t)L->L * ctx->n * L->keyw * 8)) != PG_OK) return rc;
        if ((rc = lay_alloc(ctx, L, (void **)&L->relay_val, (size_t)L->L * ctx->n * 8)) != PG_OK) return rc;
    }
    if ((rc = lay_alloc(ctx, L, (void **)&L->hist, LAY_NB * 8)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->trace, ((size_t)T + 2) * 4)) != PG_OK) return rc;
    if ((rc = lay_alloc(ctx, L, (void **)&L->d_ctrl, sizeof(LayCtrl))) != PG_OK) return rc;
    PG_CUDA(ctx, cudaMallocHost((void **)&L->h_ctrl, sizeof(LayCtrl)));
    PG_CUDA(ctx, cudaMemsetAsync(L->keys, 0, T * S * L->keyw * 8, ctx->stream));
    PG_CUDA(ctx, cudaMemsetAsync(L->vals, 0xff, T * S * 8, ctx->stream));
    PG_CUDA(ctx, cudaMemsetAsync(L->counts, 0, T * 4, ctx->stream));
    DevLay dummy;
    memset(&dummy, 0, sizeof(dummy));
    if ((rc = lay_expand(ctx, dummy, 0, true, &L->expand_grid)) != PG_OK) return rc;
    L->compact_grid = ctx->sm_count * 4;
    return PG_OK;
}

void pg_layered_close(pg_ctx *ctx, LayeredState *L)
{
    if (!L) return;
    cudaStreamSynchronize(ctx->stream);
    for (void *p : {(void *)L->keys, (void *)L->vals, (void *)L->claims, (void *)L->counts, (void *)L->list_key, (void *)L->list_val,
                    (void *)L->relay_key, (void *)L->relay_val, (void *)L->hist, (void *)L->trace, (void *)L->d_ctrl,
                    (void *)L->cand_key, (void *)L->cand_val, (void *)L->cand_f, (void *)L->sel_hist, (void *)L->ret_key,
                    (void *)L->ret_val, (void *)L->beam_trace})
        cudaFree(p);
    if (L->h_ctrl) cudaFreeHost(L->h_ctrl);
    delete L;
}

int64_t pg_layered_bytes(const LayeredState *L) { return L ? L->bytes : 0; }

int pg_layered_pass(pg_ctx *ctx, LayeredState *L, const LayPassIn &in, int64_t budget, LayPassOut &out)
{
    out = LayPassOut();
    const DevLay d = make_dev(ctx, L, in);
    if (d.nt > L->n_tables) return pg_fail(ctx, PG_ERR_STATE, "pg_search_layered: a retain pass wider than its tables");
    PG_CUDA(ctx, cudaMemsetAsync(L->d_ctrl, 0, sizeof(LayCtrl), ctx->stream));
    PG_CUDA(ctx, cudaMemsetAsync(L->hist, 0, LAY_NB * 8, ctx->stream));
    if (d.width && L->ret_cap <= 0)
        return pg_fail(ctx, PG_ERR_STATE, "pg_search_beam: the level tables were opened without a retained array");
    // the origin's low: its parent in beam mode (none), the all-ones move in retain mode, no relay yet in relay mode
    const uint32_t low0 = d.width ? ~0u : (d.retain ? (1u << d.n) - 1u : RELAY_BASE);
    if (L->keyw == 1)
        layered_seed_kernel<1><<<1, 1, 0, ctx->stream>>>(d, in.g0, low0);
    else
        layered_seed_kernel<2><<<1, 1, 0, ctx->stream>>>(d, in.g0, low0);
    PG_CUDA(ctx, cudaGetLastError());

    // levels ls .. lt - 1, checked every LAY_SYNC levels; groups of LAY_GROUP levels replay one captured graph
    const int nlev = d.lt - d.ls;
    GraphExec exec;
    bool tried = false;
    int rc = PG_OK;
    for (int done = 0; done < nlev;) {
        const int upto = std::min(nlev, done + LAY_SYNC);
        while (done < upto) {
            if (!L->no_graph && upto - done >= LAY_GROUP && nlev >= 2 * LAY_GROUP) {
                if (!tried) {
                    tried = true;
                    rc = pg_capture(ctx, [&] {
                        int e = PG_OK;
                        for (int k = 0; k < LAY_GROUP && e == PG_OK; k++) e = launch_level(ctx, L, d);
                        return e;
                    }, &exec);
                    if (rc != PG_OK) return rc;
                }
                if (exec) {
                    PG_CUDA(ctx, cudaGraphLaunch(exec.exec, ctx->stream));
                    done += LAY_GROUP;
                    continue;
                }
            }
            if ((rc = launch_level(ctx, L, d)) != PG_OK) return rc;
            done++;
        }
        if ((rc = read_ctrl(ctx, L)) != PG_OK) return rc;
        const LayCtrl &c = *L->h_ctrl;
        if (c.error) break;
        if (c.dead) break;
        if (budget > 0 && (int64_t)c.expansions >= budget) {
            out.aborted = true;
            break;
        }
    }
    // level lt: t alone (the box's last corner)
    if (!out.aborted && (rc = launch_compact(ctx, L, d, 1)) != PG_OK) return rc;
    if ((rc = read_ctrl(ctx, L)) != PG_OK) return rc;
    const LayCtrl c = *L->h_ctrl;
    if (c.error)
        return pg_fail(ctx, PG_ERR_CAPACITY, std::string(d.width ? "pg_search_beam" : "pg_search_layered") + ": a level holds more than " +
                                                 std::to_string(L->L) + " coordinates (raise table_capacity)");
    out.fmin = c.fmin;
    out.fmax = c.fmax;
    out.expansions = (int64_t)c.expansions;
    out.generated = (int64_t)c.generated;
    out.inserted = (int64_t)c.inserted;
    out.levels = (int64_t)c.levels;
    out.max_level_nodes = (int64_t)c.max_level;
    out.max_held = (int64_t)c.max_held;
    out.kept = (int64_t)c.ret_n;
    out.dropped = (int64_t)c.dropped;
    out.max_cand = (int64_t)c.max_cand;
    out.drop_fmin = c.drop_fmin;
    out.hist.assign(LAY_NB, 0);
    PG_CUDA(ctx, cudaMemcpyAsync(out.hist.data(), L->hist, LAY_NB * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (!out.aborted && !c.dead && c.d == d.lt && c.list_n == 1) {
        unsigned long long v = 0;
        PG_CUDA(ctx, cudaMemcpyAsync(&v, d.width ? L->cand_val : L->list_val, 8, cudaMemcpyDeviceToHost, ctx->stream));
        PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        out.reached = true;
        out.goal_g = (int)(v >> 32);
        out.goal_parent = (uint32_t)v;
        if (!in.retain && !d.width) {
            const uint32_t low = (uint32_t)v;
            if (low < RELAY_BASE) return pg_fail(ctx, PG_ERR_STATE, "pg_search_layered: t has no relay");
            const size_t id = low - RELAY_BASE, cap = (size_t)L->L * ctx->n;
            unsigned long long kw[2] = {0, 0}, rv = 0;
            PG_CUDA(ctx, cudaMemcpyAsync(&kw[0], L->relay_key + id, 8, cudaMemcpyDeviceToHost, ctx->stream));
            if (L->keyw == 2) PG_CUDA(ctx, cudaMemcpyAsync(&kw[1], L->relay_key + cap + id, 8, cudaMemcpyDeviceToHost, ctx->stream));
            PG_CUDA(ctx, cudaMemcpyAsync(&rv, L->relay_val + id, 8, cudaMemcpyDeviceToHost, ctx->stream));
            PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            const unsigned __int128 key = ((unsigned __int128)kw[1] << 64) | kw[0];
            const int kb = ctx->dp.key_bits;
            for (int i = 0; i < ctx->n; i++) out.relay[i] = (int)((key >> (i * kb)) & ((1u << kb) - 1u));
            out.relay_g = (int)(rv >> 32);
            out.relay_mask = (uint32_t)rv;
        }
    }
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!in.retain) { // a retain pass is cleared after its trace
        dim3 grid(std::max(1, L->compact_grid / d.nt), d.nt);
        if (L->keyw == 1)
            layered_clear_kernel<1><<<grid, LAY_THREADS, 0, ctx->stream>>>(d);
        else
            layered_clear_kernel<2><<<grid, LAY_THREADS, 0, ctx->stream>>>(d);
        PG_CUDA(ctx, cudaGetLastError());
        PG_CUDA(ctx, cudaMemsetAsync(L->counts, 0, (size_t)d.nt * 4, ctx->stream));
    }
    return PG_OK;
}

int pg_layered_trace(pg_ctx *ctx, LayeredState *L, const LayPassIn &in, std::vector<uint32_t> &masks)
{
    const DevLay d = make_dev(ctx, L, in);
    const int max_moves = d.lt - d.ls;
    if (L->keyw == 1)
        layered_trace_kernel<1><<<1, 1, 0, ctx->stream>>>(d, L->trace, max_moves);
    else
        layered_trace_kernel<2><<<1, 1, 0, ctx->stream>>>(d, L->trace, max_moves);
    PG_CUDA(ctx, cudaGetLastError());
    std::vector<uint32_t> tr((size_t)max_moves + 2);
    PG_CUDA(ctx, cudaMemcpyAsync(tr.data(), L->trace, tr.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    dim3 grid(std::max(1, L->compact_grid / d.nt), d.nt);
    if (L->keyw == 1)
        layered_clear_kernel<1><<<grid, LAY_THREADS, 0, ctx->stream>>>(d);
    else
        layered_clear_kernel<2><<<grid, LAY_THREADS, 0, ctx->stream>>>(d);
    PG_CUDA(ctx, cudaGetLastError());
    PG_CUDA(ctx, cudaMemsetAsync(L->counts, 0, (size_t)d.nt * 4, ctx->stream));
    if (tr[0] == ~0u) return pg_fail(ctx, PG_ERR_STATE, "pg_search_layered: the retained levels lost the parent chain");
    masks.resize(tr[0]);
    for (uint32_t k = 0; k < tr[0]; k++) masks[k] = tr[2 + (tr[0] - 1 - k)]; // stored t first
    return PG_OK;
}

int pg_beam_trace(pg_ctx *ctx, LayeredState *L, const LayPassIn &in, uint32_t goal_parent, std::vector<uint32_t> &masks)
{
    const DevLay d = make_dev(ctx, L, in);
    const int max_moves = d.lt - d.ls;
    if (L->keyw == 1)
        beam_trace_kernel<1><<<1, 1, 0, ctx->stream>>>(d, goal_parent, L->beam_trace, max_moves);
    else
        beam_trace_kernel<2><<<1, 1, 0, ctx->stream>>>(d, goal_parent, L->beam_trace, max_moves);
    PG_CUDA(ctx, cudaGetLastError());
    std::vector<uint32_t> tr((size_t)max_moves + 2);
    PG_CUDA(ctx, cudaMemcpyAsync(tr.data(), L->beam_trace, tr.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (tr[0] == ~0u) return pg_fail(ctx, PG_ERR_STATE, "pg_search_beam: the retained parents do not lead back to the origin");
    masks.resize(tr[0]);
    for (uint32_t k = 0; k < tr[0]; k++) masks[k] = tr[2 + (tr[0] - 1 - k)]; // stored t first
    return PG_OK;
}
