// Kernels 3+ — the batched PA-Star search: per-GPU closed/open hash table, f-indexed open buckets, and the round
// select -> claim -> expand + probe -> insert (+ the multi-GPU exchange modes), and the step-wise C ABI over them.  The
// host drivers that run whole searches on top of it are in pg_drivers.cu.
//
// Replaces, for one hash-owned partition (reference: one worker thread):
//   PAStar<N>::worker_inner      pastar/PAStar.cpp:319-401   pop / closed check / expand / reconcile
//   PAStar<N>::enqueue           pastar/PAStar.cpp:219-237   closed-list dedupe + reopen
//   PriorityList<N>              pastar/include/PriorityList.h:84-122  (pos-unique, min-f pop)
//   process_final_node/check_stop pastar/PAStar.cpp:410-547  optimality-preserving stop
//   sender / receiver / decoder  pastar/pastar_functions/*.cpp          successor exchange between partitions
//
// Data layout in HBM (all device resident, nothing per-node on the host):
//   table   ClosedList and the pos-index of OpenList in one structure: best g per coordinate.
//           The lattice is cut into aligned 2^D cubes (D = min(N, 7): the lowest bit of the first D
//           coordinates); a cube is one BLOCK of 2^D values, direct-mapped by those bits, so a value
//           needs no key of its own:
//             directory  open addressing over block keys (the packed key with those D bits cleared):
//                        KEYW=1 {u64 blockkey+1}, KEYW=2 {u64 lo, u64 hi|1<<63}; 0 = free.  Sixteen
//                        (eight) neighbouring blocks share a 128-byte directory line.
//             values     block s is values[s * 2^D ..]; VALW=4: ~(g << (N+1) | open << N | parenti) when
//                        that fits 32 bits, else VALW=8: ~(g<<32 | open<<31 | parenti); 0 = empty.
//           A successor probe reads one (L1/L2-resident) directory word and one 4-byte value: the 127
//           successors of a node touch about 30 lines of HBM instead of 54 with 16-byte keyed entries
//           (tools/microbench3.cu: a random line costs the same whatever is read from it, 36.6 G/s).
//   buckets one u64 per f value {chunk offset, log2 size, fill}: the priority index of
//           OpenList.  A bucket is a backward-linked list of chunks of u32 table slots
//           whose sizes double (64, 128, ... 256 Ki entries), so a bucket of any size
//           is a handful of contiguous runs; push = one atomicAdd, pop = whole chunks.
//   plan / live / surv   per round: chunks selected by the select kernel, parents that
//           survived the closed-bit claim, successors that passed the read-only probe.
// A round is four launches on one stream (select, claim, expand + probe, insert); every count
// that links them lives in the device control block, which the host reads every few rounds.
//
// Duplicate detection (the dominant cost): one 16 B load per successor in the expand kernel;
// 88 % of successors are rejected right there (same key, g not better) without any atomic or
// write.  The rest goes through the insert kernel: new keys take one CAS on the key word,
// improvements one CAS on the value word; only those are pushed to the open buckets.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "pg_expand_core.cuh"

namespace {

constexpr uint32_t UNIT = 64;              // pool allocation unit (table slots); first chunk of a bucket
constexpr uint32_t MAXLG = 12;             // largest chunk = UNIT << MAXLG slots
constexpr uint32_t CHUNK_NONE = 0xffffffffu;
constexpr uint32_t CNT_MASK = (1u << 27) - 1u;
// bucket state: [63:32] chunk offset in units, [31:27] log2(chunk units), [26:0] fill
__host__ __device__ constexpr unsigned long long bucket_pack(uint32_t off, uint32_t lg, uint32_t cnt)
{
    return ((unsigned long long)off << 32) | ((unsigned long long)lg << 27) | cnt;
}
constexpr unsigned long long BUCKET_EMPTY = ((unsigned long long)CHUNK_NONE << 32) | UNIT; // lg 0, "full": first push installs
constexpr int SELECT_THREADS = 1024;
constexpr int MAX_PROBE = 4096;
constexpr uint64_t OPEN_BIT = 1ull << 31;  // in the un-inverted packing

} // namespace

struct PlanEntry {
    uint32_t unit, count, offset, start; // pool[unit*UNIT + start .. +count) are batch entries offset..offset+count
};

namespace {

// ---------------------------------------------------------------------------------------------
// packed keys
// ---------------------------------------------------------------------------------------------
template <int KEYW>
struct Key;
template <>
struct Key<1> {
    unsigned long long lo;
    __device__ __forceinline__ static Key zero() { return Key{0ull}; }
    __device__ __forceinline__ void add_bit(int off) { lo += 1ull << off; }
    __device__ __forceinline__ void add_val(unsigned v, int off) { lo += (unsigned long long)v << off; }
    __device__ __forceinline__ Key plus(const Key &o) const { return Key{lo + o.lo}; }
    __device__ __forceinline__ unsigned field(int off, unsigned m) const { return (unsigned)(lo >> off) & m; }
    // 32-bit multiplicative mix of the two key halves (the directory has at most 2^28 lines); the caller takes the TOP
    // bits, which every key bit reaches: two multiplies, one xor-shift, one more multiply
    __device__ __forceinline__ unsigned long long hash() const
    {
        unsigned h = (unsigned)lo * 0x9E3779B1u + (unsigned)(lo >> 32) * 0x85EBCA77u;
        h ^= h >> 15;
        h *= 0xC2B2AE3Du;
        return h;
    }
};
template <>
struct Key<2> {
    unsigned long long lo, hi;
    __device__ __forceinline__ static Key zero() { return Key{0ull, 0ull}; }
    __device__ __forceinline__ void add_val(unsigned v, int off)
    {
        unsigned __int128 x = ((unsigned __int128)hi << 64) | lo;
        x += (unsigned __int128)v << off;
        lo = (unsigned long long)x;
        hi = (unsigned long long)(x >> 64);
    }
    __device__ __forceinline__ void add_bit(int off) { add_val(1u, off); }
    __device__ __forceinline__ Key plus(const Key &o) const
    {
        unsigned __int128 x = (((unsigned __int128)hi << 64) | lo) + (((unsigned __int128)o.hi << 64) | o.lo);
        return Key{(unsigned long long)x, (unsigned long long)(x >> 64)};
    }
    __device__ __forceinline__ unsigned field(int off, unsigned m) const
    {
        unsigned __int128 x = ((unsigned __int128)hi << 64) | lo;
        return (unsigned)(x >> off) & m;
    }
    __device__ __forceinline__ unsigned long long hash() const
    {
        unsigned h = (unsigned)lo * 0x9E3779B1u + (unsigned)(lo >> 32) * 0x85EBCA77u + (unsigned)hi * 0x165667B1u +
                     (unsigned)(hi >> 32) * 0xD3A2646Cu;
        h ^= h >> 15;
        h *= 0xC2B2AE3Du;
        return h;
    }
};


// ---------------------------------------------------------------------------------------------
// Table: block directory + direct-mapped value blocks.  A random access costs a whole 128-byte line of HBM whatever
// is read from it (36.6 G random lines/s, tools/microbench2/3.cu), so the layout minimises LINES per probe:
//   * values carry no key: the 2^D coordinates that differ only in the lowest bit of the first D coordinates form a
//     block, and a value's place inside its block is given by those D bits.  With 4-byte values a line holds a
//     5-dimensional sub-cube: the successors of a node touch 4 * 1.5^5 = 30 lines on average;
//   * the block's key is looked up in a directory that is 64 (128) times smaller than the values; neighbouring blocks
//     (lowest bit of the first four block coordinates) share a directory line, so the directory lines a frontier needs
//     stay L2 resident and a node's successors read 8 of them on average (most of them L1 hits inside a parent group).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ld_cg_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_cg_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ld_cg_v2(const unsigned long long *p, unsigned long long &a, unsigned long long &b)
{
    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void cas128(unsigned long long *addr, unsigned long long n0, unsigned long long n1, unsigned long long &o0,
                                       unsigned long long &o1)
{ // compare with {0,0}
    asm volatile(
        "{\n\t.reg .b128 c, n, o;\n\tmov.b128 c, {%3, %4};\n\tmov.b128 n, {%5, %6};\n\t"
        "atom.global.cas.b128 o, [%2], c, n;\n\tmov.b128 {%0, %1}, o;\n\t}"
        : "=l"(o0), "=l"(o1)
        : "l"(addr), "l"(0ull), "l"(0ull), "l"(n0), "l"(n1)
        : "memory");
}

struct DevSearch {
    unsigned long long *dir;      // block directory: KEYW u64 per slot
    unsigned long long dir_mask;  // directory slots - 1 (power of two)
    void *vals;                   // value blocks: (dir_mask + 1) << D values of VALW bytes
    int kb;                       // bits per coordinate in the packed key
    int D;                        // block dimensions: lowest bit of the first D coordinates
    int DL;                       // directory-line dimensions: lowest bit of the first DL BLOCK coordinates
    int nb, gs;                   // value layout: open bit position, g shift (VALW=4: N, N+1; VALW=8: 31, 32)
    int hshift;                   // 32 - log2(directory lines): the line is the top bits of the 32-bit key hash
    unsigned long long low_lo, low_hi;   // key bits that index inside a block
    unsigned long long line_lo, line_hi; // low bits + the bits that index inside a directory line
    unsigned long long *buckets;
    uint32_t *tail;
    uint32_t *hint; // per bucket: log2 units of the largest chunk it ever had
    uint32_t *pool;
    unsigned long long *link;
    uint32_t *free_stack;  // chunks popped empty by select, per size class lg at free_stack + free_off[lg]; count in ctrl->free_top[lg]
    uint32_t free_off[16];
    uint32_t n_units;
    unsigned long long goal_lo, goal_hi;
    PlanEntry *plan;
    uint32_t plan_cap;
    SearchCtrl *ctrl;
    int n_parts, part;
    char *outbox;
    unsigned long long *outbox_count;
    unsigned long long outbox_cap;
    // P2P mode: base of every partition's (peer-mapped) inbox; this partition writes region [part] of inbox[dst]
    char *peer_inbox[16];
    unsigned long long *peer_counts[16];
    int p2p;
    int f0, f_range;              // bucket 0 is f == f0; number of buckets
    // weighted search (pg_search_set_weight): h terms are floor(hnum * term >> hsh); hnum == 1: exact A*.  hrecip =
    // floor(2^32 / weight) turns a dropped successor's h_w back into a value <= its h.  goal_limit: goals (and, weighted,
    // every successor) with g >= this are dropped - the all-advance cost + 1.  inc_limit: the incumbent's cost U
    // (INT_MAX without one); a weighted successor is dropped when its lower bound g + floor(h_w * hrecip / 2^32) <= g + h
    // reaches it.  The exact search carries U in prune_limit and goal_limit alone.
    int hnum, hsh;
    unsigned hrecip;
    int goal_limit;
    int inc_limit;
    unsigned long long *live;     // compacted live parents of the round, word-major: live[w * live_cap + i]
    unsigned long long live_cap;
    unsigned long long *surv;     // local survivors of the round
    unsigned long long surv_cap;
    // expand kernel, one-word keys with at most 4 loop bits (N <= 9): key offset of every high mask, read as a constant-bank
    // operand of the add instead of a shared-memory load per successor
    unsigned long long keyhigh[16];
};

struct Counters { // per thread, flushed once per kernel
    unsigned expansions, generated, reopen, inserted, pushed, pruned, stale;
};

// ---- values.  Stored inverted, so zeroed memory is "empty, no g yet" (g reads as the largest representable).
template <int VALW>
struct ValT;
template <>
struct ValT<4> {
    typedef unsigned T;
};
template <>
struct ValT<8> {
    typedef unsigned long long T;
};
template <int VALW>
__device__ __forceinline__ typename ValT<VALW>::T val_pack(const DevSearch &d, unsigned g, unsigned mask) // an OPEN entry
{
    typedef typename ValT<VALW>::T T;
    return (T) ~(((T)g << d.gs) | ((T)1 << d.nb) | (T)mask);
}
template <int VALW>
__device__ __forceinline__ unsigned val_g(const DevSearch &d, typename ValT<VALW>::T s) // empty: larger than any real g
{
    typedef typename ValT<VALW>::T T;
    return (unsigned)((T)(~s) >> d.gs);
}
template <int VALW>
__device__ __forceinline__ bool val_closed(const DevSearch &d, typename ValT<VALW>::T s) // s != 0
{
    return (s >> d.nb) & 1;
}
template <int VALW>
__device__ __forceinline__ unsigned val_mask(const DevSearch &d, typename ValT<VALW>::T s)
{
    typedef typename ValT<VALW>::T T;
    return (unsigned)((T)(~s) & (((T)1 << d.nb) - 1));
}
// the live-parent / record form of a value: g << 32 | open << 31 | parenti
template <int VALW>
__device__ __forceinline__ unsigned long long val_record(const DevSearch &d, typename ValT<VALW>::T s, bool open)
{
    return ((unsigned long long)val_g<VALW>(d, s) << 32) | (open ? OPEN_BIT : 0ull) | (unsigned long long)val_mask<VALW>(d, s);
}
template <int VALW>
__device__ __forceinline__ typename ValT<VALW>::T *val_ptr(const DevSearch &d, unsigned long long slot)
{
    return reinterpret_cast<typename ValT<VALW>::T *>(d.vals) + slot;
}
template <int VALW>
__device__ __forceinline__ typename ValT<VALW>::T ld_val(const typename ValT<VALW>::T *p)
{
    if constexpr (VALW == 4)
        return ld_cg_u32(p);
    else
        return ld_cg_u64(p);
}

// asynchronous 4 / 8-byte copy global -> shared: the value load of a probe holds no register while it is in flight
template <int BYTES>
__device__ __forceinline__ void cp_async_val(void *smem, const void *gmem)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    if constexpr (BYTES == 4)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa), "l"(gmem) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// ---- keys -> block key, place inside the block, directory slot
template <int KEYW>
__device__ __forceinline__ Key<KEYW> block_key(const DevSearch &d, const Key<KEYW> &key)
{
    Key<KEYW> b = key;
    b.lo &= ~d.low_lo;
    if constexpr (KEYW == 2) b.hi &= ~d.low_hi;
    return b;
}
// index of `key` inside its block: the lowest bit of the first D coordinates
template <int KEYW>
__device__ __forceinline__ unsigned block_index(const DevSearch &d, const Key<KEYW> &key)
{
    unsigned idx = 0;
    for (int i = 0; i < d.D; i++) idx |= key.field(i * d.kb, 1u) << i;
    return idx;
}
// the key of entry `idx` of the block `bkey`
template <int KEYW>
__device__ __forceinline__ Key<KEYW> block_entry_key(const DevSearch &d, Key<KEYW> bkey, unsigned idx)
{
    for (int i = 0; i < d.D; i++)
        if ((idx >> i) & 1u) bkey.add_bit(i * d.kb);
    return bkey;
}
// place of a block inside its directory line: the lowest bit of the first DL block coordinates (bit 1 of the coordinates)
template <int KEYW>
__device__ __forceinline__ unsigned dir_pos(const DevSearch &d, const Key<KEYW> &key)
{
    unsigned idx = 0;
    for (int i = 0; i < d.DL; i++) idx |= key.field(i * d.kb + 1, 1u) << i;
    return idx;
}
template <int KEYW>
constexpr int DIR_LB = KEYW == 1 ? 4 : 3; // log2 directory slots per 128-byte line
// home directory slot of the block that holds `key`; dpos = dir_pos(key)
template <int KEYW>
__device__ __forceinline__ unsigned long long dir_home(const DevSearch &d, const Key<KEYW> &key, unsigned dpos)
{
    Key<KEYW> lk = key;
    lk.lo &= ~d.line_lo;
    if constexpr (KEYW == 2) lk.hi &= ~d.line_hi;
    return (((lk.hash() >> d.hshift) << DIR_LB<KEYW>) | dpos) & d.dir_mask; // top bits of the multiplicative hash pick the line
}
template <int KEYW>
__device__ __forceinline__ unsigned long long dir_next(const DevSearch &d, unsigned long long dslot)
{
    return (dslot + (1ull << DIR_LB<KEYW>)) & d.dir_mask;
}
template <int KEYW>
__device__ __forceinline__ bool dir_is(const unsigned long long h0, const unsigned long long h1, const Key<KEYW> &bkey)
{
    if constexpr (KEYW == 1)
        return h0 == bkey.lo + 1;
    else
        return h0 == bkey.lo && h1 == (bkey.hi | (1ull << 63));
}

// Find the directory slot of the block `bkey`, starting at `dslot`; claim a free slot when `claim`.  Returns the slot
// or ~0 (absent when !claim, directory full when claim).
template <int KEYW>
__device__ __forceinline__ unsigned long long dir_find(const DevSearch &d, const Key<KEYW> &bkey, unsigned long long dslot, bool claim)
{
    for (int probe = 0; probe < MAX_PROBE; probe++, dslot = dir_next<KEYW>(d, dslot)) {
        unsigned long long *e = d.dir + dslot * KEYW;
        unsigned long long h0, h1 = 0;
        if constexpr (KEYW == 1)
            h0 = ld_cg_u64(e);
        else
            ld_cg_v2(e, h0, h1);
        if (dir_is<KEYW>(h0, h1, bkey)) return dslot;
        if (h0 != 0 || h1 != 0) continue;
        if (!claim) return ~0ull;
        if constexpr (KEYW == 1) {
            const unsigned long long prev = atomicCAS(e, 0ull, bkey.lo + 1);
            if (prev == 0 || prev == bkey.lo + 1) return dslot;
        } else {
            unsigned long long p0, p1;
            cas128(e, bkey.lo, bkey.hi | (1ull << 63), p0, p1);
            if ((p0 == 0 && p1 == 0) || dir_is<KEYW>(p0, p1, bkey)) return dslot;
        }
    }
    return ~0ull;
}
// value slot (index into d.vals) of `key`, or ~0
template <int KEYW>
__device__ __forceinline__ unsigned long long table_find(const DevSearch &d, const Key<KEYW> &key, bool claim)
{
    const Key<KEYW> bkey = block_key<KEYW>(d, key);
    const unsigned long long dslot = dir_find<KEYW>(d, bkey, dir_home<KEYW>(d, key, dir_pos<KEYW>(d, key)), claim);
    if (dslot == ~0ull) return ~0ull;
    return (dslot << d.D) | block_index<KEYW>(d, key);
}

// Push a table slot on the open bucket of f.  One atomicAdd hands out a position:
//   old fill < capacity : the slot is written in place (the fast path; callers may issue the atomic themselves and
//                         pass its result to bucket_place, so that several pushes are in flight per thread)
//   old fill == capacity: this thread installs the next (twice as large) chunk
//   old fill > capacity : an install is in flight; poll until the new head is published, then retry
__device__ __noinline__ void bucket_place_slow(const DevSearch &d, int b, uint32_t slot, unsigned long long st)
{
    SearchCtrl *c = d.ctrl;
    unsigned long long *bk = d.buckets + b;
    for (;;) {
        const uint32_t cnt = (uint32_t)st & CNT_MASK, lg = ((uint32_t)st >> 27) & 31u, off = (uint32_t)(st >> 32);
        const uint32_t capn = UNIT << lg;
        if (cnt < capn) {
            d.pool[(size_t)off * UNIT + cnt] = slot;
            return;
        }
        if (cnt == capn) {
            // First chunk of a (re)filled bucket: as large as the bucket grew last time (d.hint), so a hot bucket is
            // not re-grown 64, 128, ... every round.  Pushers that lost the race poll until the new head is published,
            // so the critical section is only bump + publish; bookkeeping that only the select kernel reads comes after.
            const uint32_t nlg = off == CHUNK_NONE ? min(d.hint[b], MAXLG) : min(lg + 1u, MAXLG);
            // a chunk the select kernel popped empty (this round's claim kernel has read it: inserts run after it), else fresh
            // pool space.  Pops only race with pops (select, the only pusher, never runs beside an insert kernel).
            uint32_t nc;
            const int ft = atomicSub(&c->free_top[nlg], 1) - 1;
            if (ft >= 0) {
                nc = d.free_stack[d.free_off[nlg] + ft];
            } else {
                atomicAdd(&c->free_top[nlg], 1);
                nc = atomicAdd(&c->chunk_bump, 1u << nlg);
                if ((unsigned long long)nc + (1u << nlg) > d.n_units) {
                    c->error = 2;
                    atomicExch(bk, bucket_pack(off, lg, capn)); // leave the bucket consistent
                    return;
                }
            }
            atomicExch(bk, bucket_pack(nc, nlg, 1u));
            d.link[nc] = ((unsigned long long)off << 32) | lg;
            d.pool[(size_t)nc * UNIT] = slot;
            if (off != CHUNK_NONE) atomicAdd(&d.tail[b], capn);
            if (nlg > d.hint[b]) d.hint[b] = nlg;
            return;
        }
        for (;;) { // install in flight
            const unsigned long long cur = ld_cg_u64(bk);
            if (((uint32_t)cur & CNT_MASK) <= (UNIT << (((uint32_t)cur >> 27) & 31u))) break;
        }
        st = atomicAdd(bk, 1ull);
    }
}
// bucket index of f, or -1 (error raised) when f is beyond the bucket range
__device__ __forceinline__ int bucket_of(const DevSearch &d, int f)
{
    const int b = f - d.f0; // f0 / f_range are constants of the search: read from the kernel parameters, not from the control
                            // block whose line is busy with counter atomics
    if (b < 0) { // f below h(start): the heuristic is not consistent for this cost model; reported, never clamped
        d.ctrl->error = 5;
        return -1;
    }
    if (b >= d.f_range) {
        d.ctrl->error = 3;
        return -1;
    }
    return b;
}
__device__ __forceinline__ void bucket_place(const DevSearch &d, int b, uint32_t slot, unsigned long long st)
{
    const uint32_t cnt = (uint32_t)st & CNT_MASK, lg = ((uint32_t)st >> 27) & 31u, off = (uint32_t)(st >> 32);
    if (cnt < (UNIT << lg))
        d.pool[(size_t)off * UNIT + cnt] = slot;
    else
        bucket_place_slow(d, b, slot, st);
}
__device__ __forceinline__ void bucket_push(const DevSearch &d, int f, uint32_t slot)
{
    const int b = bucket_of(d, f);
    if (b < 0) return;
    bucket_place(d, b, slot, atomicAdd(d.buckets + b, 1ull));
}

// ---------------------------------------------------------------------------------------------
// select: pick the chunks to pop this round (one CTA)
// ---------------------------------------------------------------------------------------------
// Inclusive scan of a[] and b2[] over the SELECT_THREADS (= 32 warps x 32) threads of the CTA, in place: shuffles inside
// a warp, the 32 warp totals scanned by warp 0, three barriers in all.
__device__ __forceinline__ void block_scan2(unsigned *a, unsigned *b2, int t)
{
    __shared__ unsigned s_wa[32], s_wb[32];
    const int lane = t & 31, w = t >> 5;
    unsigned x = a[t], y = b2[t];
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned vx = __shfl_up_sync(0xffffffffu, x, off), vy = __shfl_up_sync(0xffffffffu, y, off);
        if (lane >= off) {
            x += vx;
            y += vy;
        }
    }
    if (lane == 31) {
        s_wa[w] = x;
        s_wb[w] = y;
    }
    __syncthreads();
    if (w == 0) {
        unsigned tx = s_wa[lane], ty = s_wb[lane];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned vx = __shfl_up_sync(0xffffffffu, tx, off), vy = __shfl_up_sync(0xffffffffu, ty, off);
            if (lane >= off) {
                tx += vx;
                ty += vy;
            }
        }
        s_wa[lane] = tx;
        s_wb[lane] = ty;
    }
    __syncthreads();
    if (w > 0) {
        x += s_wa[w - 1];
        y += s_wb[w - 1];
    }
    a[t] = x;
    b2[t] = y;
    __syncthreads();
}

__global__ void __launch_bounds__(SELECT_THREADS) select_kernel(DevSearch d, long long target, int f_limit)
{
    __shared__ unsigned s_a[SELECT_THREADS];
    __shared__ unsigned s_b[SELECT_THREADS];
    __shared__ int s_first;
    SearchCtrl *c = d.ctrl;
    const int t = threadIdx.x;
    if (t == 0) {
        c->batch_n = 0;
        c->plan_n = 0;
        if (target > 0) { // a status-only select (target 0) leaves the round's lists alone
            c->live_n = 0;
            c->surv_n = 0;
        }
    }
    if (target > 0 && d.n_parts > 1 && t < d.n_parts) d.outbox_count[t] = 0;
    if (c->done || c->error) return;
    const int range = c->f_range;
    const int limit_f = min(f_limit, c->best_goal);
    const long long limit_b = (long long)limit_f - c->f0; // buckets >= limit_b are not popped
    // ---- first non-empty bucket at or after the cursor
    int cursor = c->cursor;
    int first = -1;
    while (cursor < range) {
        if (t == 0) s_first = INT_MAX;
        __syncthreads();
        const int b = cursor + t;
        if (b < range && (uint32_t)(d.buckets[b] >> 32) != CHUNK_NONE) atomicMin(&s_first, b);
        __syncthreads();
        first = s_first;
        __syncthreads();
        if (first != INT_MAX) break;
        cursor += SELECT_THREADS;
        first = -1;
    }
    if (first < 0) { // open list exhausted
        if (t == 0) {
            c->cursor = range;
            c->min_open_f = INT_MAX;
            if (d.n_parts == 1) c->done = 2;
        }
        return;
    }
    if (t == 0) {
        c->cursor = first;
        c->min_open_f = c->f0 + first;
    }
    if ((long long)first >= limit_b) { // every open node has f >= best goal (or the caller's limit)
        if (t == 0 && d.n_parts == 1 && c->best_goal != INT_MAX && first >= c->best_goal - c->f0) c->done = 1;
        return;
    }
    // ---- window of SELECT_THREADS buckets starting at `first`
    const int b = first + t;
    unsigned entries = 0, cnt = 0, lg = 0, off = CHUNK_NONE;
    if (b < range && (long long)b < limit_b) {
        const unsigned long long st = d.buckets[b];
        off = (uint32_t)(st >> 32);
        if (off != CHUNK_NONE) {
            lg = ((uint32_t)st >> 27) & 31u;
            cnt = min((uint32_t)st & CNT_MASK, UNIT << lg);
            entries = cnt + d.tail[b];
        }
    }
    s_a[t] = entries;
    s_b[t] = 0;
    __syncthreads();
    block_scan2(s_a, s_b, t);
    const unsigned before = s_a[t] - entries;
    __syncthreads();
    // A bucket is taken if the buckets before it did not reach the target; the one that
    // crosses it gives exactly the missing entries, newest first (chunks are stacks: the
    // top of the head chunk is popped and its fill lowered).
    unsigned take_chunks = 0, take_entries = 0;
    if (entries && (long long)before < target) {
        const unsigned want = (unsigned)min((long long)entries, target - before);
        take_entries = want;
        take_chunks = 1;
        unsigned got = min(cnt, want);
        unsigned long long lk = d.link[off];
        while (got < want) {
            got += UNIT << (uint32_t)(lk & 31u);
            take_chunks++;
            lk = d.link[(uint32_t)(lk >> 32)];
        }
    }
    s_a[t] = take_entries;
    s_b[t] = take_chunks;
    __syncthreads();
    block_scan2(s_a, s_b, t);
    unsigned e_off = s_a[t] - take_entries;
    const unsigned p_off = s_b[t] - take_chunks;
    const unsigned total_e = s_a[SELECT_THREADS - 1], total_p = s_b[SELECT_THREADS - 1];
    if (total_p > d.plan_cap) {
        if (t == 0) c->error = 2;
        return;
    }
    if (take_chunks) {
        uint32_t ch = off, chlg = lg;
        unsigned left = take_entries, fill = cnt, remain = entries;
        for (unsigned i = 0;; i++) {
            const unsigned n = min(fill, left);
            d.plan[p_off + i] = PlanEntry{ch, n, e_off, fill - n}; // entries [fill-n, fill) of the chunk
            e_off += n;
            left -= n;
            remain -= n;
            if (n == fill) { // popped empty: the bucket lets go of it; recycled by this round's inserts (after the claim kernel)
                const int ft = atomicAdd(&c->free_top[chlg], 1);
                d.free_stack[d.free_off[chlg] + ft] = ch;
            }
            if (n < fill || remain == 0) { // this chunk keeps fill-n entries and stays the head
                fill -= n;
                break;
            }
            const unsigned long long lk = d.link[ch];
            ch = (uint32_t)(lk >> 32);
            chlg = (uint32_t)(lk & 31u);
            fill = UNIT << chlg;
            if (left == 0) break; // next chunk untouched: it becomes a full head
        }
        if (remain == 0) {
            d.buckets[b] = BUCKET_EMPTY;
            d.tail[b] = 0;
        } else {
            d.buckets[b] = bucket_pack(ch, chlg, fill);
            d.tail[b] = remain - fill;
        }
    }
    if (t == 0) {
        c->batch_n = (int)total_e;
        c->plan_n = (int)total_p;
        c->pops += total_e;
    }
}

// One record at a time: find / claim the block of `key` starting at directory slot `dslot`, install g if strictly
// better, push.  Returns UPS_* flags.
enum { UPS_INSERTED = 1, UPS_PUSHED = 2, UPS_REOPEN = 4 };
template <int KEYW, int VALW>
__device__ __noinline__ unsigned upsert_from(const DevSearch &d, const Key<KEYW> key, unsigned long long dslot, int gnew, int f, int mask)
{
    typedef typename ValT<VALW>::T T;
    unsigned flags = 0;
    dslot = dir_find<KEYW>(d, block_key<KEYW>(d, key), dslot, true);
    if (dslot == ~0ull) {
        d.ctrl->error = 1;
        return flags;
    }
    const unsigned long long slot = (dslot << d.D) | block_index<KEYW>(d, key);
    T *vp = val_ptr<VALW>(d, slot);
    T val = ld_val<VALW>(vp);
    const T mine = val_pack<VALW>(d, (unsigned)gnew, (unsigned)mask);
    for (;;) {
        if ((unsigned)gnew >= val_g<VALW>(d, val)) return flags; // PAStar.cpp:228 / PriorityList.h:109: not better, drop
        const T prev = atomicCAS(vp, val, mine);
        if (prev == val) break;
        val = prev;
    }
    if (val == 0)
        flags |= UPS_INSERTED;
    else if (val_closed<VALW>(d, val))
        flags |= UPS_REOPEN; // was closed with a worse g: PAStar.cpp:230-231
    bucket_push(d, f, (uint32_t)slot);
    return flags | UPS_PUSHED;
}

// ---------------------------------------------------------------------------------------------
// the search round: select -> claim -> expand + probe -> insert
// ---------------------------------------------------------------------------------------------
// claim   one thread per popped open-list entry: plan lookup, closed-bit claim (PAStar.cpp:344-351).  Entries
//         that are stale (a better g was pushed later) or already closed drop out here; the live parents are
//         compacted into d.live, so the expansion only sees nodes that are really expanded and needs no barrier.
// expand  a group of 2^A lanes per live parent, no CTA-wide synchronisation in the loop: LUT / HH staging
//         (pg_expand_prepare), then per lane
//            pass 1: f, g, key, owner and home slot of its next successors; ISSUE all their table loads (up to 8
//                    independent 16 B loads in flight per lane);
//            pass 2: compare.  The common case (same key, g not better: PAStar.cpp:228 / PriorityList.h:109)
//                    ends here: the kernel only READS the table.  Survivors - new key, better g, hash collision -
//                    are appended to the
//                    round's survivor list.  Successors owned by another partition go to that partition's outbox
//                    (or straight into its peer-mapped inbox over NVLink) unprobed: the owner filters them.
// insert  survivors and records received from other partitions: CAS on key / value, push to the f bucket
//         (PAStar.cpp:219-237 enqueue, PriorityList.h:104-113 conditional_enqueue), 4 records in flight per thread.
#ifdef PG_PHASE_TIMING
#define PH_MARK(idx) do { long long t__ = clock64(); ph[idx] += t__ - ph_t; ph_t = t__; } while (0)
#else
#define PH_MARK(idx) do { } while (0)
#endif

// Owner hash arguments.  Z-order hashes (SURVEY F5): bit m of the owner word is bit `bit[m]` of coordinate `co[m]`
// (co < 0: beyond the coordinate width, reads 0); the word is reduced mod n_parts through a 256-entry table.
struct OwnerArgs {
    int type, shift, nb;
    int co[8], bit[8];
    int nfc;            // distinct coordinates the owner word reads ...
    int fc[8], fcm[8];  // ... and, per coordinate, the mask of owner-word bits tied to it
};

// The round's parents as the expand kernel sees them: one or more word-major regions ((KEYW + 1) arrays of `cap`
// u64: key words, then ~value) whose record counts live in device memory.  own = 0: parents forwarded by other
// partitions (their owners count the expansion).
struct ParentSrc {
    const unsigned long long *base[16];
    const unsigned long long *count[16];
    unsigned long long cap;
    int n;
    unsigned own; // bit r: region r holds this partition's own parents
};

// Partitions (bit set) that own at least one successor of the node `key`; `part` itself is not reported.
template <int KEYW>
__device__ __forceinline__ unsigned successor_owners(const DevProblem &p, const OwnerArgs &oa, const Key<KEYW> &key, int n_parts, int part)
{
    const unsigned fmask = (1u << p.key_bits) - 1u;
    unsigned set = 0;
    if (oa.type == PG_HASH_FSUM || oa.type == PG_HASH_PSUM) {
        const int nd = oa.type == PG_HASH_PSUM ? 2 : p.n;
        unsigned sum = 0;
        int movable = 0, others = 0;
        for (int i = 0; i < p.n; i++) {
            const unsigned pc = key.field(i * p.key_bits, fmask);
            if (i < nd) {
                sum += pc;
                movable += (int)pc < p.len[i];
            } else {
                others += (int)pc < p.len[i];
            }
        }
        for (int k = others ? 0 : 1; k <= movable; k++) set |= 1u << (((sum + k) >> oa.shift) % (unsigned)n_parts);
    } else {
        unsigned wbase = 0, delta[8];
        for (int k = 0; k < oa.nfc; k++) {
            const int co = oa.fc[k];
            const unsigned pc = key.field(co * p.key_bits, fmask);
            unsigned dl = 0;
            for (int m = 0; m < oa.nb; m++) {
                if (!((oa.fcm[k] >> m) & 1)) continue;
                const unsigned v0 = (pc >> oa.bit[m]) & 1u, v1 = ((pc + 1u) >> oa.bit[m]) & 1u;
                wbase |= v0 << m;
                dl |= (v0 ^ v1) << m;
            }
            delta[k] = (int)pc < p.len[co] ? dl : 0u; // a sequence at its end does not move (borderCheck, Node.cpp:69-77)
        }
        for (int sset = 0; sset < (1 << oa.nfc); sset++) {
            unsigned w = wbase;
            bool real = true;
            for (int k = 0; k < oa.nfc; k++)
                if ((sset >> k) & 1) {
                    w ^= delta[k];
                    real = real && delta[k] != 0; // moving a coordinate that changes nothing is the same class
                }
            if (real) set |= 1u << (w % (unsigned)n_parts);
        }
    }
    return set & ~(1u << part);
}

constexpr int STAMP_SHIFT = 40; // counts stay below 2^40; the bits above carry the exchange round + 1 (data-flow synchronisation)
constexpr unsigned long long COUNT_MASK = (1ull << STAMP_SHIFT) - 1ull;
constexpr uint32_t PROBE_MISS = 0xffffffffu;        // stash: the probe found no block of its own at the home directory slot
constexpr unsigned long long HINT_FLAG = 1ull << 31; // record word KEYW+1: {start slot : 32 | HINT_FLAG | move mask : 16}
constexpr int RING_CAP = 64;                         // insert kernel: deferred-record ring, items per warp
constexpr int PLAN_SM = 2048;

template <int KEYW, int VALW>
__global__ void __launch_bounds__(256) claim_kernel(const __grid_constant__ DevSearch d)
{
    typedef typename ValT<VALW>::T T;
#ifndef PG_CLAIM_PF
#define PG_CLAIM_PF 1 // 4 / 2 / 1 pops per thread: 58 / 51 / 48 us - with one pop per thread the batch is 3.5 waves of CTAs whose
                      // phases (pool read, value line, atomic) overlap instead of every thread of one wave marching through them in step
#endif
    constexpr int PF = PG_CLAIM_PF; // pops per thread, each step of their dependent chains (plan -> pool -> table) issued for all of them
    __shared__ uint32_t s_plan[PLAN_SM];
    __shared__ int s_wtot[8];
    __shared__ unsigned long long s_base;
    SearchCtrl *c = d.ctrl;
    __shared__ int s_batch_n;
    if (threadIdx.x == 0) s_batch_n = (c->done || c->error) ? 0 : c->batch_n; // read once per CTA: barriers follow
    __syncthreads();
    const int batch_n = s_batch_n;
    if (batch_n == 0) return;
    const int plan_n = c->plan_n;
    const bool plan_sm = plan_n <= PLAN_SM;
    if (plan_sm)
        for (int i = threadIdx.x; i < plan_n; i += blockDim.x) s_plan[i] = d.plan[i].offset;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    for (int base = blockIdx.x * 256 * PF; base < batch_n; base += gridDim.x * 256 * PF) {
        int bi[PF], pl[PF];
        uint32_t slot[PF];
        T old[PF];
        unsigned long long klo[PF], khi[PF];
#pragma unroll
        for (int j = 0; j < PF; j++) {
            bi[j] = base + j * 256 + threadIdx.x;
            int lo = 0, hi = plan_n - 1;
            if (bi[j] < batch_n) {
                while (lo < hi) { // last plan entry with offset <= bi
                    const int mid = (lo + hi + 1) >> 1;
                    const uint32_t off = plan_sm ? s_plan[mid] : d.plan[mid].offset;
                    if ((int)off <= bi[j])
                        lo = mid;
                    else
                        hi = mid - 1;
                }
            }
            pl[j] = lo;
        }
#pragma unroll
        for (int j = 0; j < PF; j++) {
            slot[j] = 0;
            if (bi[j] < batch_n) {
                const PlanEntry pe = d.plan[pl[j]];
                slot[j] = d.pool[(size_t)pe.unit * UNIT + pe.start + (bi[j] - pe.offset)];
            }
        }
#pragma unroll
        for (int j = 0; j < PF; j++) {
            old[j] = (T)1 << d.nb; // "already closed": not live
            klo[j] = khi[j] = 0;
            // Three of four popped entries are stale (the node was closed through a better entry): a plain load of the
            // value decides those - ONE random line, where the atomic plus the block's key cost two and a write-back.
            if (bi[j] < batch_n) old[j] = ld_val<VALW>(val_ptr<VALW>(d, slot[j]));
        }
#pragma unroll
        for (int j = 0; j < PF; j++) {
            if (!val_closed<VALW>(d, old[j])) {
                // mark closed: set the (inverted) open bit; whoever sees it clear owns the expansion (PAStar.cpp:344-351).
                // The block's key never changes once the block exists, so it is read alongside.
                old[j] = atomicOr(val_ptr<VALW>(d, slot[j]), (T)1 << d.nb);
                const unsigned long long *e = d.dir + (size_t)(slot[j] >> d.D) * KEYW;
                klo[j] = ld_cg_u64(e);
                if constexpr (KEYW == 2) khi[j] = ld_cg_u64(e + 1);
            }
        }
        // compaction: one atomic on the live counter per CTA sweep (a per-warp atomic on that single address was 60 % of
        // this kernel's stall samples): warp totals -> shared-memory prefix -> one reservation for the CTA
        unsigned bal[PF];
        int wtot = 0;
#pragma unroll
        for (int j = 0; j < PF; j++) {
            bal[j] = __ballot_sync(0xffffffffu, !val_closed<VALW>(d, old[j]));
            wtot += __popc(bal[j]);
        }
        if (lane == 0) s_wtot[threadIdx.x >> 5] = wtot;
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < 8; w++) {
                const int t = s_wtot[w];
                s_wtot[w] = tot;
                tot += t;
            }
            s_base = tot ? atomicAdd(&c->live_n, (unsigned long long)tot) : 0ull;
        }
        __syncthreads();
        unsigned long long wbase = s_base + (unsigned long long)s_wtot[threadIdx.x >> 5];
        __syncthreads(); // s_wtot / s_base are rewritten by the next sweep
#pragma unroll
        for (int j = 0; j < PF; j++) {
            if (!val_closed<VALW>(d, old[j])) {
                Key<KEYW> bkey;
                bkey.lo = KEYW == 1 ? klo[j] - 1 : klo[j];
                if constexpr (KEYW == 2) bkey.hi = khi[j] & ~(1ull << 63);
                const Key<KEYW> key = block_entry_key<KEYW>(d, bkey, slot[j] & ((1u << d.D) - 1u));
                unsigned long long *r = d.live + (size_t)(wbase + __popc(bal[j] & lt));
                r[0] = key.lo;
                if constexpr (KEYW == 2) r[d.live_cap] = key.hi;
                r[KEYW * d.live_cap] = val_record<VALW>(d, old[j], true);
            }
            wbase += __popc(bal[j]);
        }
    }
}

// Parent forwarding (multi-GPU): every partition that owns a successor of a live parent gets the parent itself (16 or
// 24 bytes over NVLink, stored straight into its peer-mapped inbox) and generates its own successors from it, instead
// of receiving them one by one.  One thread per live parent; one counter atomic per (warp, destination).
template <int KEYW>
__global__ void __launch_bounds__(256) forward_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevSearch d,
                                                      const __grid_constant__ OwnerArgs oa)
{
    SearchCtrl *c = d.ctrl;
    const int lane = threadIdx.x & 31;
    {   // warp-uniform early exit (c->error may be raised by another CTA of this launch; ballots follow)
        int skip = lane == 0 ? (c->done || c->error) : 0;
        if (__shfl_sync(0xffffffffu, skip, 0)) return;
    }
    const long long live_n = (long long)c->live_n;
    const unsigned lt = (1u << lane) - 1u;
    for (long long base = (long long)blockIdx.x * 256; base < live_n; base += (long long)gridDim.x * 256) {
        const long long i0 = base + threadIdx.x;
        unsigned owners = 0;
        unsigned long long klo = 0, khi = 0, val = 0;
        if (i0 < live_n) {
            klo = d.live[i0];
            if constexpr (KEYW == 2) khi = d.live[d.live_cap + i0];
            val = d.live[KEYW * d.live_cap + i0];
            Key<KEYW> key;
            key.lo = klo;
            if constexpr (KEYW == 2) key.hi = khi;
            owners = successor_owners<KEYW>(p, oa, key, d.n_parts, d.part);
        }
        for (int dst = 0; dst < d.n_parts; dst++) {
            const unsigned b = __ballot_sync(0xffffffffu, (owners >> dst) & 1u);
            if (!b) continue;
            unsigned long long base0 = 0;
            if (lane == __ffs(b) - 1) base0 = atomicAdd(&d.outbox_count[dst], (unsigned long long)__popc(b));
            base0 = __shfl_sync(0xffffffffu, base0, __ffs(b) - 1);
            if ((owners >> dst) & 1u) {
                const unsigned long long i = base0 + __popc(b & lt);
                if (i < d.outbox_cap) {
                    unsigned long long *r = reinterpret_cast<unsigned long long *>(d.peer_inbox[dst]) + (size_t)d.part * d.outbox_cap * (KEYW + 1) + i;
                    r[0] = klo;
                    if constexpr (KEYW == 2) r[d.outbox_cap] = khi;
                    r[KEYW * d.outbox_cap] = val;
                } else {
                    c->error = 4;
                }
            }
        }
    }
}

// Outbox space is handed out in chunks of OBOX_CHUNK records per (CTA, destination): one global atomic per chunk,
// shared-memory atomics inside it.  state = {first record of the chunk : 40 | records used : 24}.  Records a chunk
// does not use are marked as holes (move mask 0) and skipped by the receiver.
constexpr unsigned OBOX_CHUNK = 256;
// Where record `pos` for partition dst lives: the local outbox (NCCL all-to-all mode), or directly the owner's
// peer-mapped inbox over NVLink (P2P mode): region [this partition] of inbox[dst].
template <int KEYW>
__device__ __forceinline__ unsigned long long *outbox_record(const DevSearch &d, int dst, unsigned long long pos)
{
    constexpr int XW = KEYW == 1 ? 3 : 4;
    if (d.p2p) return reinterpret_cast<unsigned long long *>(d.peer_inbox[dst]) + ((size_t)d.part * d.outbox_cap + pos) * XW;
    return reinterpret_cast<unsigned long long *>(d.outbox) + ((size_t)dst * d.outbox_cap + pos) * XW;
}
template <int KEYW>
__device__ __forceinline__ void outbox_mark_holes(const DevSearch &d, int dst, unsigned long long base, unsigned from)
{
    constexpr int XW = KEYW == 1 ? 3 : 4;
    unsigned long long *r = outbox_record<KEYW>(d, dst, base);
    for (unsigned i = from; i < OBOX_CHUNK; i++) r[(size_t)i * XW + KEYW + 1] = 0ull;
}
template <int KEYW>
__device__ __noinline__ unsigned long long outbox_reserve(const DevSearch &d, unsigned long long *s_obox, int dst, int k)
{
    for (;;) {
        const unsigned long long st = atomicAdd(&s_obox[dst], (unsigned long long)k);
        const unsigned used = (unsigned)(st & 0xffffffull);
        const unsigned long long base = st >> 24;
        if (used + k <= OBOX_CHUNK) return base + used;
        if (used <= OBOX_CHUNK) { // first to run over the chunk: close it and open the next one
            if (used < OBOX_CHUNK) outbox_mark_holes<KEYW>(d, dst, base, used);
            unsigned long long nb = atomicAdd(&d.outbox_count[dst], (unsigned long long)OBOX_CHUNK);
            if (nb + OBOX_CHUNK > d.outbox_cap) {
                d.ctrl->error = 4;
                nb = 0; // keep writes in bounds; the run is abandoned with PG_ERR_CAPACITY
            }
            atomicExch(&s_obox[dst], nb << 24);
        } else { // another warp is opening the next chunk
            while (((*(volatile unsigned long long *)&s_obox[dst]) >> 24) == base &&
                   ((*(volatile unsigned long long *)&s_obox[dst]) & 0xffffffull) > OBOX_CHUNK) { }
        }
    }
}

// MODE 0: one partition.  MODE 1: successors owned by other partitions are sent to them as records.  MODE 2: they are
// skipped - their owners generate them from the forwarded parent (claim_kernel<.., true>).
#ifndef PG_EXPAND_CTAS
#define PG_EXPAND_CTAS 3 // resident CTAs per SM the expand kernel is compiled for (register budget 65536 / 256 / this)
#endif
// LOOPOWN = false: the owner hash reads only coordinates that are lane bits (PZORDER, PSUM, FZORDER with its bits in the
// first A coordinates), so a lane's successors all have one owner and the per-successor owner arithmetic is not compiled.
template <int N, int KEYW, int VALW, int MODE, bool LOOPOWN = true>
__global__ void __launch_bounds__(256, PG_EXPAND_CTAS) expand_probe_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevSearch d,
                                                              const __grid_constant__ OwnerArgs oa, const __grid_constant__ ParentSrc ps)
{
    constexpr bool MULTI = MODE != 0;   // owners are computed
    constexpr bool SEND = MODE == 1;    // ... and records sent
    typedef typename ValT<VALW>::T T;
    using C = ExpCfg<N>;
    constexpr int XW = KEYW == 1 ? 3 : 4;
    constexpr int GROUPS = 256 / C::LP;
    constexpr int GPW = 32 / C::LP; // parent groups per warp
    constexpr int NI = 1 << C::IB;
#ifdef PG_PFMAX
    constexpr int PFMAX = PG_PFMAX;
#else
    constexpr int PFMAX = (KEYW == 1 && N < 14) ? 8 : 4; // N >= 14: the HH tables leave less shared memory for the stash
#endif
    constexpr int PF = NI < PFMAX ? NI : PFMAX; // successors whose table loads are in flight together, per lane
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PairMeta *meta = reinterpret_cast<PairMeta *>(smem_raw);
    Key<KEYW> *s_keyhigh = reinterpret_cast<Key<KEYW> *>(smem_raw + ((sizeof(PairMeta) + 15) & ~size_t(15)));
    int *s_groups = reinterpret_cast<int *>(s_keyhigh + C::H);
    // probe stash: what the deferred compare of a batch needs, [PF][256] each, a thread only touches its own column
    T *s_pv = reinterpret_cast<T *>(s_groups + GROUPS * C::GROUP_INTS);      // values (cp.async destination)
    int *s_pg = reinterpret_cast<int *>(s_pv + PF * 256);                    // g
    int *s_pf = s_pg + PF * 256;                                             // f
    uint32_t *s_ps = reinterpret_cast<uint32_t *>(s_pf + PF * 256);          // directory slot, PROBE_MISS when the block was not at its home slot
    __shared__ unsigned long long s_cnt[4];
    __shared__ unsigned long long s_obox[SEND ? 64 : 1];
    __shared__ unsigned char s_mod[MULTI ? 256 : 1]; // owner word -> partition
    __shared__ int s_droplb[256];                    // weighted search: this thread's min of g + h over its dropped successors

    SearchCtrl *c = d.ctrl;
    // the flags are read ONCE per CTA (other CTAs of this launch may raise c->error while this one starts; the warps of a
    // CTA must agree on the early return because barriers follow)
    __shared__ int s_skip;
    if (threadIdx.x == 0) {
        unsigned long long any = 0;
        for (int rg = 0; rg < ps.n; rg++) any |= *ps.count[rg] & COUNT_MASK;
        s_skip = (c->done || c->error || any == 0) ? 1 : 0;
    }
    __syncthreads();
    if (s_skip) return;
    const int prune = c->prune_limit;
    const int best0 = c->best_goal;
    const int limit = min(prune, best0);

    pg_load_pair_meta(p, meta);
    for (int hi = threadIdx.x; hi < C::H; hi += blockDim.x) {
        Key<KEYW> k = Key<KEYW>::zero();
        for (int b = 0; b < C::HB; b++)
            if ((hi >> b) & 1) k.add_bit((C::A + b) * p.key_bits);
        s_keyhigh[hi] = k;
    }
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    s_droplb[threadIdx.x] = INT_MAX;
    if (SEND && threadIdx.x < 64) s_obox[threadIdx.x] = (unsigned long long)OBOX_CHUNK; // no chunk yet: the first append opens one
    if (MULTI) s_mod[threadIdx.x & 255] = (unsigned char)((threadIdx.x & 255) % (unsigned)d.n_parts);
    __syncthreads();

    // key offset of a high mask: a kernel parameter where the table is small (see DevSearch::keyhigh), else shared memory
    auto keyhi = [&](int high) -> Key<KEYW> {
        if constexpr (KEYW == 1 && C::HB <= 4) {
            return Key<KEYW>{d.keyhigh[high]};
        } else {
            return s_keyhigh[high];
        }
    };
    const int grp = threadIdx.x / C::LP, sub = threadIdx.x % C::LP;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned gmask = C::LP == 32 ? 0xffffffffu : (((1u << C::LP) - 1u) << (lane & ~(C::LP - 1)));
    const unsigned lt = (1u << lane) - 1u;
    int *s_grp = s_groups + grp * C::GROUP_INTS;
    const int *s_hhg = s_grp + 8 * C::P;
    const int *s_hhh = s_hhg + C::H;
#ifdef PG_PHASE_TIMING
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long ph_t = clock64();
#endif
    unsigned n_exp = 0, n_gen = 0, n_pruned = 0;
    const unsigned fmask = (1u << p.key_bits) - 1u;
    const int full = (1 << N) - 1;

    // ---- owner hash, split into what is fixed for the kernel, per lane, and per parent.  Z-order hashes (SURVEY F5): bit m of
    // the owner word is bit oa.bit[m] of coordinate oa.co[m].  lanemask = the word bits whose coordinate this LANE moves,
    // hmask[b] = the word bits of the coordinate the b-th loop bit moves.  Sum hashes: the successor's sum is the parent's
    // plus the number of moved sequences among the first nd.
    unsigned lanemask = 0, hmask[C::HB > 0 ? C::HB : 1];
#pragma unroll
    for (int b = 0; b < C::HB; b++) hmask[b] = 0;
    const bool zorder = oa.type != PG_HASH_FSUM && oa.type != PG_HASH_PSUM;
    const int sum_nd = oa.type == PG_HASH_PSUM ? 2 : N;
    const int ksub = __popc(sub & ((1 << sum_nd) - 1)); // sum hashes: sequences this lane moves (N >= 3 > 2: PSUM is lane-uniform)
    if constexpr (MULTI) {
        if (zorder) {
            for (int m = 0; m < oa.nb; m++) {
                const int co = oa.co[m];
                if (co < 0) continue;
                if (co < C::A) {
                    if ((sub >> co) & 1) lanemask |= 1u << m;
                } else {
#pragma unroll
                    for (int b = 0; b < C::HB; b++)
                        if (co - C::A == b) hmask[b] |= 1u << m;
                }
            }
        }
    }

    // ---- the deferred half of a probe batch: compare the values that have arrived; stage the survivors
    bool pend = false;          // warp-uniform
    unsigned pend_vmask = 0;    // which of the batch's PF probes this lane issued
    int pend_hb = 0;            // high-mask index of the batch's first probe
    Key<KEYW> pend_klow = Key<KEYW>::zero();
    auto complete = [&]() {
        cp_async_wait_all();
        // same coordinate, g not better (PAStar.cpp:228 / PriorityList.h:109) ends here: the common case.  A probe that
        // found no block of its own left an empty value (g = infinity) in the stash.
        unsigned slowmask = 0;
#pragma unroll
        for (int j = 0; j < PF; j++) {
            const int gn = s_pg[j * 256 + threadIdx.x];
            const bool slow = ((pend_vmask >> j) & 1u) && (unsigned)gn < val_g<VALW>(d, s_pv[j * 256 + threadIdx.x]);
            slowmask |= (slow ? 1u : 0u) << j;
        }
        // The batch's survivors (one in eight) go straight to the round's survivor list: one warp-wide prefix sum over the
        // lanes' counts and one atomic per batch.  (Round 1-2a staged them in a per-warp shared-memory ring: a ballot, an
        // append, a __syncwarp and a flush test per successor, and 12 KB of shared memory per CTA that the L1 now has:
        // 380 -> 336 us.)
        const unsigned mine = __popc(slowmask);
        unsigned incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
        if (total) { // warp-uniform
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(&c->surv_n, (unsigned long long)total);
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base + total > d.surv_cap) {
                c->error = 4;
            } else {
                unsigned long long *q = d.surv + (base + (incl - mine)) * XW;
#pragma unroll
                for (int j = 0; j < PF; j++) {
                    if ((slowmask >> j) & 1u) {
                        const uint32_t hit = s_ps[j * 256 + threadIdx.x];
                        const int high = pend_hb + j;
                        const Key<KEYW> key = pend_klow.plus(keyhi(high));
                        q[0] = key.lo;
                        if constexpr (KEYW == 2) q[1] = key.hi;
                        q[KEYW] = ((unsigned long long)(unsigned)s_pg[j * 256 + threadIdx.x] << 32) | (unsigned)s_pf[j * 256 + threadIdx.x];
                        // the directory slot is a hint for the insert kernel when this successor's block was found there
                        q[KEYW + 1] = (hit != PROBE_MISS ? ((unsigned long long)hit << 32) | HINT_FLAG : 0ull) | (unsigned long long)(unsigned)((high << C::A) | sub);
                        q += XW;
                    }
                }
            }
        }
        pend = false;
        PH_MARK(4); // pass 2: wait for the probes, compare, stage
    };

    // parents are dealt to the groups round-robin; the trip count is warp-uniform (the ring is a warp-level structure)
    const int stride = gridDim.x * GROUPS;
    for (int rg = 0; rg < ps.n; rg++) {
    const unsigned long long *live = ps.base[rg];
    const int live_n = (int)min(*ps.count[rg] & COUNT_MASK, ps.cap);
    int pi = blockIdx.x * GROUPS + grp;
    unsigned long long nk0 = 0, nk1 = 0, nval = 0;
    if (pi < live_n) {
        const unsigned long long *r = live + (size_t)pi;
        nk0 = __ldg(r);
        if constexpr (KEYW == 2) nk1 = __ldg(r + ps.cap);
        nval = __ldg(r + KEYW * ps.cap);
    }
    // (a dynamic deal of the parents - GPW at a time from a counter, the next deal's atomic in flight during the expansion -
    // measured the same 381 us as this static round-robin: the groups' 13-or-14-parents tail is not what the launch waits for)
    for (int wfirst = blockIdx.x * GROUPS + warp * GPW; wfirst < live_n; wfirst += stride, pi += stride) {
        bool act = pi < live_n;
        Key<KEYW> pkey = Key<KEYW>::zero();
        pkey.lo = nk0;
        if constexpr (KEYW == 2) pkey.hi = nk1;
        const unsigned long long val = nval;
        if (pi + stride < live_n) { // the next parent's record travels while this one is expanded
            const unsigned long long *r = live + (size_t)(pi + stride);
            nk0 = __ldg(r);
            if constexpr (KEYW == 2) nk1 = __ldg(r + ps.cap);
            nval = __ldg(r + KEYW * ps.cap);
        }
        int pos[N];
        int goal_mask = 0;
        ExpLane<N> L;
        L.alive = 0;
        if (act) {
            const int g = (int)(unsigned)(val >> 32), parenti = (int)(val & 0xffffu);
            int alive = 0, onestep = 0;
#pragma unroll
            for (int i = 0; i < N; i++) {
                pos[i] = (int)pkey.field(i * p.key_bits, fmask);
                alive |= (pos[i] < p.len[i]) << i;
                onestep |= (pos[i] + 1 == p.len[i]) << i;
            }
            if (alive == 0) {
                act = false; // the goal itself: never expanded (PAStar.cpp:353-357)
            } else {
                // the goal is reached from here by moving every sequence that is one short of its end
                goal_mask = alive == onestep ? alive : 0;
                if (sub == 0 && ((ps.own >> rg) & 1u)) n_exp++;
                pg_expand_prepare<N>(p, meta, s_grp, pos, g, parenti, sub, gmask, L, d.hnum, d.hsh);
            }
        }
        unsigned wbase = 0, wany = 0;
        unsigned wflip[C::HB > 0 ? C::HB : 1];
#pragma unroll
        for (int b = 0; b < C::HB; b++) wflip[b] = 0;
        int qmod = 0, rk = 0; // sum hashes: (parent sum >> shift) % n_parts, low part of the sum + this lane's moves
        bool uniform = false; // one owner for all of this lane's successors
        if constexpr (MULTI) {
            if (zorder) {
                unsigned w0 = 0, w1 = 0; // owner word with no / every owner coordinate advanced
                for (int m = 0; m < oa.nb; m++) {
                    const int co = oa.co[m];
                    if (co < 0) continue;
                    const unsigned pc = pkey.field(co * p.key_bits, fmask);
                    w0 |= ((pc >> oa.bit[m]) & 1u) << m;
                    w1 |= (((pc + 1u) >> oa.bit[m]) & 1u) << m;
                }
                wbase = (w0 & ~lanemask) | (w1 & lanemask);
                if constexpr (LOOPOWN) {
#pragma unroll
                    for (int b = 0; b < C::HB; b++) {
                        wflip[b] = (w0 ^ w1) & hmask[b];
                        wany |= wflip[b];
                    }
                }
                uniform = wany == 0; // most parents lie inside one partition's cell in every loop coordinate
            } else {
                unsigned psum = 0;
#pragma unroll
                for (int i = 0; i < N; i++)
                    if (i < sum_nd) psum += act ? (unsigned)pos[i] : 0u;
                qmod = (int)((psum >> oa.shift) % (unsigned)d.n_parts);
                rk = (int)(psum & ((1u << oa.shift) - 1u)) + ksub;
                const int kmax = sum_nd > C::A ? sum_nd - C::A : 0; // loop bits that count towards the sum
                uniform = !LOOPOWN || ((unsigned)rk >> oa.shift) == ((unsigned)(rk + kmax) >> oa.shift);
                wbase = (unsigned)qmod + ((unsigned)rk >> oa.shift); // < 64 + 17: s_mod reduces it
            }
        }
        const int lown = uniform ? (int)s_mod[wbase] : d.part;
        const bool own_all = uniform && lown == d.part;
        const bool own_none = MODE == 2 && uniform && lown != d.part;
        const bool lane_foreign = SEND && act && uniform && lown != d.part; // MODE 1: the lane's whole batch goes to partition lown
        PH_MARK(2); // prepare (LUT gathers, HH, B/E)
        Key<KEYW> klow = pkey;
#pragma unroll
        for (int i = 0; i < C::A; i++)
            if ((sub >> i) & 1) klow.add_bit(i * p.key_bits);
        const bool interior = L.alive == full;
        // A successor's place inside its block is the parent's low bits XOR the move mask (adding 1 flips the lowest
        // bit); a block coordinate moves on where the parent's low bit is set and the sequence advances.
        unsigned plow = 0, pdir = 0;
        if (act) {
#pragma unroll
            for (int i = 0; i < N; i++) {
                if (i < d.D) plow |= (unsigned)(pos[i] & 1) << i;
                if (i < d.DL) pdir |= (unsigned)((pos[i] >> 1) & 1) << i;
            }
        }
        const unsigned bem = (1u << d.D) - 1u, dlm = (1u << d.DL) - 1u;

        for (int u = 0; u < (1 << C::UB); u++) {
            int vg[NI], vh[NI];
            pg_expand_block<N>(L, u, vg, vh);
#pragma unroll
            for (int cb = 0; cb < NI; cb += PF) {
                // the previous batch (of this parent, or the last one of the previous parent: its value loads travelled
                // while this parent's LUTs were staged) is compared before its stash is reused
                if (pend) complete();
                // MODE 1, lane-uniform owner: the lanes of a warp that send to the same partition reserve their PF record
                // slots each with ONE atomic on that destination's counter; a lane then stores its records (a hole for
                // a successor that does not exist or is pruned) straight into the owner's inbox while it computes
                unsigned long long *obase = nullptr;
                if constexpr (SEND) {
                    const unsigned fl = __ballot_sync(0xffffffffu, lane_foreign);
                    if (lane_foreign) {
                        const unsigned grp = __match_any_sync(fl, lown);
                        const int leader = __ffs(grp) - 1;
                        const unsigned long long k = (unsigned long long)__popc(grp) * PF;
                        unsigned long long b0 = 0;
                        if (lane == leader) {
                            b0 = atomicAdd(&d.outbox_count[lown], k);
                            if (b0 + k > d.outbox_cap) {
                                c->error = 4;
                                b0 = 0; // keep writes in bounds; the run is abandoned with PG_ERR_CAPACITY
                            }
                        }
                        b0 = __shfl_sync(grp, b0, leader);
                        obase = outbox_record<KEYW>(d, lown, b0 + (unsigned long long)__popc(grp & lt) * PF);
                    }
                }
                unsigned long long h0[PF], h1[KEYW == 2 ? PF : 1]; // directory words
                uint32_t ls[PF];                                     // directory slots
                unsigned vmask = 0;
                // ---- pass 1a: f, pruning, owner; ISSUE the directory loads (L1 / L2: neighbouring successors share words)
#pragma unroll
                for (int j = 0; j < PF; j++) {
                    const int i = cb + j;
                    const int high = (u << C::IB) | i;
                    const int mask = (high << C::A) | sub;
                    bool v = act && mask != 0 && (interior || !(mask & ~L.alive));
                    bool rem = false;
                    int rown = 0, gn = 0, fn = 0;
                    h0[j] = 0;
                    if constexpr (KEYW == 2) h1[j] = 0;
                    ls[j] = 0;
                    int own = d.part;
                    if constexpr (MODE == 2) v = v && !own_none;
                    if constexpr (MULTI) {
                        if (LOOPOWN && v && !own_all && !lane_foreign) {
                            if (!zorder) {
                                // the successor's sum is the parent's plus the sequences moved: (sum >> shift) % n_parts
                                const int kh = sum_nd > C::A ? __popc((unsigned)high & ((1u << (sum_nd - C::A)) - 1u)) : 0;
                                own = (int)s_mod[(unsigned)qmod + ((unsigned)(rk + kh) >> oa.shift)];
                            } else {
                                // the owner word of a successor differs from wbase (this lane, no high move) only in the
                                // bits tied to the high coordinates that move: one XOR per moved coordinate
                                unsigned w = wbase;
#pragma unroll
                                for (int b = 0; b < C::HB; b++)
                                    if ((high >> b) & 1) w ^= wflip[b];
                                own = (int)s_mod[w];
                            }
                            if (MODE == 2 && own != d.part) v = false; // its owner generates it from the forwarded parent
                        }
                    }
                    if (v) {
                        gn = vg[i] + s_hhg[high];
                        fn = gn + vh[i] + s_hhh[high];
                        n_gen++;
                        const bool is_goal = mask == goal_mask;
                        // a goal (f == g) beyond the upper bound can never be optimal - UB is the cost of a valid
                        // alignment - and one worse than the best goal known is useless: both are dropped like any
                        // other successor, so nothing past the bucket range is ever pushed
                        bool drop = fn >= limit;
                        if (is_goal) {
                            drop = gn >= d.goal_limit || gn > best0;
                            if (!drop) atomicMin(&c->best_goal, gn);
                        } else if (d.hnum > 1) {
                            // weighted: f_w no longer bounds g, so g beyond the all-advance cost is dropped as well; what
                            // the f_w test drops may still lie on an optimal path - its g + h is kept for the lower bound.
                            // With an incumbent, a successor whose bound reaches its cost U cannot lead to a cheaper one.
                            const int lbn = gn + (int)(((unsigned long long)(unsigned)(fn - gn) * d.hrecip) >> 32);
                            drop = drop || gn >= d.goal_limit || lbn >= d.inc_limit;
                            if (drop)
                                s_droplb[threadIdx.x] = min(s_droplb[threadIdx.x], lbn);
                        }
                        if (drop) {
                            n_pruned++;
                            v = false;
                        }
                    }
                    if constexpr (SEND) {
                        if (obase) { // lane-uniform owner elsewhere: record j of this lane's reservation (move mask 0 = hole)
                            unsigned long long *r = obase + j * XW;
                            const Key<KEYW> key = klow.plus(keyhi(high));
                            r[0] = key.lo;
                            if constexpr (KEYW == 2) r[1] = key.hi;
                            r[KEYW] = ((unsigned long long)(unsigned)gn << 32) | (unsigned)fn;
                            r[KEYW + 1] = v ? (unsigned long long)(unsigned)mask : 0ull;
                            v = false;
                        }
                    }
                    if (v) {
                        if constexpr (SEND) {
                            if (own != d.part) { // remote successor: goes to the owner's outbox below
                                rem = true;
                                rown = own;
                                v = false;
                            }
                        }
                        if (v) {
                            const Key<KEYW> key = klow.plus(keyhi(high));
                            const unsigned dpos = (pdir ^ (plow & (unsigned)mask)) & dlm;
                            const unsigned long long dslot = dir_home<KEYW>(d, key, dpos);
                            ls[j] = (uint32_t)dslot;
                            const unsigned long long *e = d.dir + dslot * KEYW;
                            if constexpr (KEYW == 1) {
                                h0[j] = __ldg(e);
                            } else {
                                const ulonglong2 hh = __ldg(reinterpret_cast<const ulonglong2 *>(e));
                                h0[j] = hh.x;
                                h1[j] = hh.y;
                            }
                            s_pg[j * 256 + threadIdx.x] = gn;
                            s_pf[j * 256 + threadIdx.x] = fn;
                            vmask |= 1u << j;
                        }
                    }
                    if constexpr (SEND) { // one reservation per (warp, destination) from the CTA's outbox chunks
                        unsigned todo = __ballot_sync(0xffffffffu, rem);
                        while (todo) {
                            const int leader = __ffs(todo) - 1;
                            const int dst = __shfl_sync(0xffffffffu, rown, leader);
                            const unsigned same = __ballot_sync(0xffffffffu, rem && rown == dst);
                            unsigned long long pos0 = 0;
                            if (lane == leader) pos0 = outbox_reserve<KEYW>(d, s_obox, dst, __popc(same));
                            pos0 = __shfl_sync(0xffffffffu, pos0, leader);
                            if (rem && rown == dst) {
                                unsigned long long *r = outbox_record<KEYW>(d, dst, pos0 + __popc(same & lt));
                                const Key<KEYW> key = klow.plus(keyhi(high));
                                r[0] = key.lo;
                                if constexpr (KEYW == 2) r[1] = key.hi;
                                r[KEYW] = ((unsigned long long)(unsigned)gn << 32) | (unsigned)fn;
                                r[KEYW + 1] = (unsigned long long)(unsigned)mask;
                            }
                            todo &= ~same;
                        }
                    }
                }
                // ---- pass 1b: where the directory word is this successor's block, ISSUE the 4 / 8-byte value load as an
                //      asynchronous copy into the stash (it holds no register while it travels).  No block there (free slot:
                //      nothing of this cube exists yet) or another block's key (collision): the successor goes to the
                //      insert kernel, which walks the directory.
#pragma unroll
                for (int j = 0; j < PF; j++) {
                    if ((vmask >> j) & 1u) {
                        const int i = cb + j;
                        const int high = (u << C::IB) | i;
                        const int mask = (high << C::A) | sub;
                        const Key<KEYW> bkey = block_key<KEYW>(d, klow.plus(keyhi(high)));
                        unsigned long long w1 = 0;
                        if constexpr (KEYW == 2) w1 = h1[j];
                        uint32_t hit = PROBE_MISS;
                        if (dir_is<KEYW>(h0[j], w1, bkey)) {
                            const unsigned idx = (plow ^ (unsigned)mask) & bem;
                            cp_async_val<VALW>(s_pv + j * 256 + threadIdx.x, val_ptr<VALW>(d, ((unsigned long long)ls[j] << d.D) | idx));
                            hit = ls[j];
                        } else {
                            s_pv[j * 256 + threadIdx.x] = 0; // "empty": the deferred compare sends it on
                        }
                        s_ps[j * 256 + threadIdx.x] = hit;
                    }
                }
                cp_async_commit();
                pend = true;
                pend_vmask = vmask;
                pend_hb = (u << C::IB) | cb;
                pend_klow = klow;
                PH_MARK(3); // pass 1: issue probes (+ remote appends)
            }
        }
        __syncwarp(); // the group's LUTs are rewritten by the next parent
    }
    } // parent regions
    if (pend) complete();
    PH_MARK(5);
#ifdef PG_PHASE_TIMING
    if (lane == 0)
        for (int k = 0; k < 8; k++) atomicAdd(&c->phase[k], (unsigned long long)ph[k]);
#endif

    // ---- close the CTA's open outbox chunks
    if constexpr (SEND) {
        __syncthreads();
        if ((int)threadIdx.x < d.n_parts) {
            const unsigned long long st = s_obox[threadIdx.x];
            const unsigned used = (unsigned)(st & 0xffffffull);
            if (used < OBOX_CHUNK) outbox_mark_holes<KEYW>(d, threadIdx.x, st >> 24, used);
        }
    }
    // ---- counters: one atomic per CTA per counter
    {
        unsigned v[3] = {n_exp, n_gen, n_pruned};
#pragma unroll
        for (int k = 0; k < 3; k++) {
            unsigned x = v[k];
            for (int o = 16; o; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
            if (lane == 0 && x) atomicAdd(&s_cnt[k], (unsigned long long)x);
        }
    }
    if (d.hnum > 1) {
        const int m = __reduce_min_sync(0xffffffffu, s_droplb[threadIdx.x]);
        if (lane == 0 && m != INT_MAX) atomicMin(&c->drop_lb, m);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicAdd(&c->expansions, s_cnt[0]);
        atomicAdd(&c->generated, s_cnt[1]);
        atomicAdd(&c->pruned, s_cnt[2]);
    }
}

// Dedupe + push of successor records: the round's local survivors and the records received from other partitions
// (PAStar.cpp:240-250 consume_queue -> enqueue; PAStar.cpp:219-237; PriorityList.h:104-113).  The record count is read
// from device memory, so a driver can chain rounds without a host round trip.  Every step of the chain
//     record -> directory word (-> claim a free slot for a new block) -> value -> CAS value (strictly better g)
//            -> bucket atomicAdd -> pool store
// runs for one record per thread at a time (PG_INS_PF): the warps of the 8 resident CTAs per SM drift apart, so their phases overlap.
// What does not fit the straight line (directory collision, a CAS lost to a concurrent writer, a bucket whose chunk is
// full) takes the one-record-at-a-time path (upsert_from / bucket_place_slow).
#ifndef PG_INS_CTAS
#define PG_INS_CTAS 4
#endif
template <int KEYW, int VALW>
__global__ void __launch_bounds__(256, PG_INS_CTAS) insert_kernel(const __grid_constant__ DevSearch d, const unsigned long long *__restrict__ recs,
                                                        const unsigned long long *__restrict__ n_ptr, unsigned long long n_max)
{
    typedef typename ValT<VALW>::T T;
    constexpr int XW = KEYW == 1 ? 3 : 4;
#ifndef PG_INS_PF
#define PG_INS_PF 1
#endif
    constexpr int PF = PG_INS_PF; // records in flight per thread.  The kernel sits at the rate of random HBM transactions (one cold value line per record):
                          // 1 / 2 / 4 / 8 in flight measured 158 / 162 / 175 / 260 us, a three-stage software pipeline (loads of two batches in flight while a
                          // third does its atomics) 159 us - profiles/r02_experiments.md
    enum { DONE = 0, DIR = 1, VAL = 2, PUSH = 3, WALK = 4 };
    SearchCtrl *c = d.ctrl;
    {   // warp-uniform early exit: other CTAs of this launch may raise c->error, and warp-level ballots follow
        int skip = (threadIdx.x & 31) == 0 ? c->error : 0;
        if (__shfl_sync(0xffffffffu, skip, 0)) return;
    }
    const long long n = (long long)min(*n_ptr & COUNT_MASK, n_max);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&c->table_used, (unsigned long long)n); // records seen by insert kernels
    Counters cn = {0, 0, 0, 0, 0, 0, 0};
    int min_b = INT_MAX;
    const int prune = c->prune_limit;
    const int limit = min(prune, c->best_goal);
    __shared__ unsigned long long s_walk[8 * RING_CAP * XW];
    __shared__ int s_droplb[256]; // weighted search: this thread's min of g + h over the records it dropped
    s_droplb[threadIdx.x] = INT_MAX;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    unsigned long long *wq = s_walk + (size_t)(threadIdx.x >> 5) * RING_CAP * XW;
    unsigned qhead = 0, qtail = 0; // warp-uniform
    auto walk_one = [&](const unsigned long long *it) {
        Key<KEYW> k;
        k.lo = it[0];
        if constexpr (KEYW == 2) k.hi = it[1];
        const unsigned long long g_f = it[KEYW], m = it[KEYW + 1];
        const unsigned fl = upsert_from<KEYW, VALW>(d, k, m >> 32, (int)(unsigned)(g_f >> 32), (int)(unsigned)g_f, (int)(m & 0xffffu));
        cn.inserted += fl & UPS_INSERTED;
        cn.pushed += (fl >> 1) & 1u;
        cn.reopen += (fl >> 2) & 1u;
        if (fl & UPS_PUSHED) min_b = min(min_b, (int)(unsigned)g_f - d.f0);
    };
    const long long stride = (long long)gridDim.x * blockDim.x;
    // the trip count is warp-uniform: the deferred ring is a warp-level structure
    for (long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x; i0 - lane < n; i0 += stride * PF) {
        Key<KEYW> key[PF], bkey[PF];
        unsigned long long gf[PF], h0[PF], h1[KEYW == 2 ? PF : 1];
        T lv[PF], lo[PF];
        uint32_t st[PF]; // directory slot
        unsigned mk[PF];
        int state[PF];
        // ---- records
#pragma unroll
        for (int j = 0; j < PF; j++) {
            const long long i = i0 + j * stride;
            state[j] = DONE;
            key[j] = Key<KEYW>::zero();
            bkey[j] = Key<KEYW>::zero();
            gf[j] = 0;
            mk[j] = 0;
            st[j] = 0;
            h0[j] = 0;
            lv[j] = lo[j] = 0;
            if (i < n) {
                const unsigned long long *r = recs + i * XW;
                key[j].lo = __ldcs(r);
                if constexpr (KEYW == 2) key[j].hi = __ldcs(r + 1);
                gf[j] = __ldcs(r + KEYW);
                const unsigned long long m = __ldcs(r + KEYW + 1);
                mk[j] = (unsigned)m & 0xffffu;
                st[j] = (uint32_t)(m >> 32);
                state[j] = mk[j] == 0 ? DONE : ((m & HINT_FLAG) ? VAL : DIR); // move mask 0: hole left by the sender's chunked outbox
            }
        }
        // ---- goal / pruning; directory words of the records that carry no directory slot
#pragma unroll
        for (int j = 0; j < PF; j++) {
            if (state[j] == DONE) continue;
            bool is_goal = key[j].lo == d.goal_lo;
            if constexpr (KEYW == 2) is_goal = is_goal && key[j].hi == d.goal_hi;
            bool drop = (int)(unsigned)gf[j] >= limit;
            if (is_goal) { // kept iff within the upper bound and at least as good as every goal seen so far (f == g)
                const int gg = (int)(unsigned)(gf[j] >> 32);
                drop = gg >= d.goal_limit || gg > atomicMin(&c->best_goal, gg);
            } else if (d.hnum > 1) { // as in the expand kernel
                const int gg = (int)(unsigned)(gf[j] >> 32);
                drop = drop || gg >= d.goal_limit;
                if (drop)
                    s_droplb[threadIdx.x] = min(s_droplb[threadIdx.x], gg + (int)(((unsigned long long)((unsigned)gf[j] - (unsigned)gg) * d.hrecip) >> 32));
            }
            if (drop) {
                state[j] = DONE;
                continue;
            }
            bkey[j] = block_key<KEYW>(d, key[j]);
            if (state[j] == DIR) {
                st[j] = (uint32_t)dir_home<KEYW>(d, key[j], dir_pos<KEYW>(d, key[j]));
                const unsigned long long *e = d.dir + (size_t)st[j] * KEYW;
                if constexpr (KEYW == 1)
                    h0[j] = ld_cg_u64(e);
                else
                    ld_cg_v2(e, h0[j], h1[j]);
            }
        }
        // ---- resolve the block: found, or claim the free slot (a new block: its values are all empty)
#pragma unroll
        for (int j = 0; j < PF; j++) {
            if (state[j] != DIR) continue;
            unsigned long long w1 = 0;
            if constexpr (KEYW == 2) w1 = h1[j];
            if (dir_is<KEYW>(h0[j], w1, bkey[j])) {
                state[j] = VAL;
            } else if (h0[j] == 0 && w1 == 0) {
                unsigned long long *e = d.dir + (size_t)st[j] * KEYW;
                unsigned long long p0, p1 = 0;
                if constexpr (KEYW == 1)
                    p0 = atomicCAS(e, 0ull, bkey[j].lo + 1);
                else
                    cas128(e, bkey[j].lo, bkey[j].hi | (1ull << 63), p0, p1);
                state[j] = ((p0 == 0 && p1 == 0) || dir_is<KEYW>(p0, p1, bkey[j])) ? VAL : WALK; // lost the slot to another block: walk on
            } else {
                state[j] = WALK; // collision: the walk continues from the next line
                st[j] = (uint32_t)dir_next<KEYW>(d, st[j]);
            }
        }
        // ---- values
        uint32_t vs[PF]; // value slot
#pragma unroll
        for (int j = 0; j < PF; j++) {
            vs[j] = 0;
            if (state[j] != VAL) continue;
            vs[j] = (uint32_t)(((unsigned long long)st[j] << d.D) | block_index<KEYW>(d, key[j]));
            lv[j] = ld_val<VALW>(val_ptr<VALW>(d, vs[j]));
        }
        // ---- CAS the value where this record is strictly better (lv = the value the CAS expects, lo = what it found)
#pragma unroll
        for (int j = 0; j < PF; j++) {
            if (state[j] != VAL) continue;
            const unsigned gnew = (unsigned)(gf[j] >> 32);
            if (gnew >= val_g<VALW>(d, lv[j])) {
                state[j] = DONE; // not better: drop (PAStar.cpp:228 / PriorityList.h:109)
                continue;
            }
            lo[j] = atomicCAS(val_ptr<VALW>(d, vs[j]), lv[j], val_pack<VALW>(d, gnew, mk[j]));
        }
        // ---- bucket positions for the records that went in
        int bk[PF];
        unsigned long long bst[PF];
#pragma unroll
        for (int j = 0; j < PF; j++) {
            bk[j] = -1;
            bst[j] = 0;
            if (state[j] != VAL) continue;
            if (lo[j] == lv[j]) {
                if (lv[j] == 0)
                    cn.inserted++;
                else if (val_closed<VALW>(d, lv[j]))
                    cn.reopen++; // was closed with a worse g: PAStar.cpp:230-231
                cn.pushed++;
                bk[j] = bucket_of(d, (int)(unsigned)gf[j]);
                state[j] = bk[j] >= 0 ? PUSH : DONE;
                if (bk[j] >= 0) {
                    min_b = min(min_b, bk[j]);
                    bst[j] = atomicAdd(d.buckets + bk[j], 1ull);
                }
            } else {
                // a concurrent writer changed the value: still better than what is there now?
                state[j] = (unsigned)(gf[j] >> 32) < val_g<VALW>(d, lo[j]) ? WALK : DONE;
            }
        }
#pragma unroll
        for (int j = 0; j < PF; j++)
            if (state[j] == PUSH) bucket_place(d, bk[j], vs[j], bst[j]);
        // ---- everything else goes to the warp's deferred ring and is handled 32 at a time with every lane busy (about
        //      1 % of the records: done in place, one straggling lane would stall its warp in most iterations)
#pragma unroll
        for (int j = 0; j < PF; j++) {
            const unsigned wb = __ballot_sync(0xffffffffu, state[j] == WALK);
            if (!wb) continue;
            if (state[j] == WALK) {
                unsigned long long *q = wq + (size_t)((qtail + __popc(wb & lt)) & (RING_CAP - 1)) * XW;
                q[0] = key[j].lo;
                if constexpr (KEYW == 2) q[1] = key[j].hi;
                q[KEYW] = gf[j];
                q[KEYW + 1] = ((unsigned long long)st[j] << 32) | (unsigned long long)mk[j];
            }
            qtail += __popc(wb);
            __syncwarp();
            if (qtail - qhead >= 32u) {
                walk_one(wq + (size_t)((qhead + lane) & (RING_CAP - 1)) * XW);
                qhead += 32u;
                __syncwarp();
            }
        }
    }
    if (lane < (int)(qtail - qhead)) walk_one(wq + (size_t)((qhead + lane) & (RING_CAP - 1)) * XW);
    // A node may have a lower f than anything open here (it came from another partition, or this partition's open
    // list ran empty): pull the select cursor back so the next round sees it.
    for (int o = 16; o; o >>= 1) min_b = min(min_b, __shfl_down_sync(0xffffffffu, min_b, o));
    if ((threadIdx.x & 31) == 0 && min_b != INT_MAX) atomicMin(&c->cursor, max(min_b, 0));
    if (d.hnum > 1) {
        const int m = __reduce_min_sync(0xffffffffu, s_droplb[threadIdx.x]);
        if (lane == 0 && m != INT_MAX) atomicMin(&c->drop_lb, m);
    }
    unsigned v[3] = {cn.inserted, cn.pushed, cn.reopen};
#pragma unroll
    for (int k = 0; k < 3; k++)
        for (int o = 16; o; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
    if ((threadIdx.x & 31) == 0) {
        if (v[0]) atomicAdd(&c->inserted, (unsigned long long)v[0]);
        if (v[1]) atomicAdd(&c->pushed, (unsigned long long)v[1]);
        if (v[2]) atomicAdd(&c->reopen, (unsigned long long)v[2]);
    }
}

// P2P mode: tell every owner how many records this partition stored into its inbox this round.
__global__ void publish_counts_kernel(const __grid_constant__ DevSearch d, int stamped)
{
    const int dst = threadIdx.x;
    const unsigned long long stamp = stamped ? d.ctrl->xround + 1ull : 0ull;
    if (dst < d.n_parts && d.peer_counts[dst]) {
        __threadfence_system(); // the records / parents this count covers were stored by earlier kernels of this stream
        d.peer_counts[dst][d.part] = (stamp << STAMP_SHIFT) | d.outbox_count[dst];
    }
}
// Device-side wait for the other partitions' counts of this exchange round (replaces a cross-GPU barrier: a count is
// written after the data it covers, and a partition cannot run more than one round ahead because its next round waits
// for this partition's next stamp).  One thread per source; gives up after ~20 s (a peer failed) with an error.  The
// round counter lives in the control block and moves on here.
__global__ void wait_counts_kernel(const __grid_constant__ DevSearch d)
{
    const int src = threadIdx.x;
    const unsigned long long stamp = d.ctrl->xround + 1ull;
    __syncthreads(); // every thread has read the counter before thread 0 moves it on
    if (src < d.n_parts && src != d.part) {
        const volatile unsigned long long *slot = d.peer_counts[d.part] + src;
        const long long t0 = clock64();
        while ((*slot >> STAMP_SHIFT) < stamp) {
            if (clock64() - t0 > 40000000000ll) {
                d.ctrl->error = 6;
                break;
            }
        }
        __threadfence_system();
    }
    __syncthreads();
    if (threadIdx.x == 0) d.ctrl->xround = stamp;
}


// Seed: insert the start node (Sequences::get_initial_node, Sequences.cpp:70-77; PAStar.cpp:153).
template <int KEYW, int VALW>
__global__ void seed_kernel(const __grid_constant__ DevSearch d, int f, int parenti)
{
    const Key<KEYW> key = Key<KEYW>::zero();
    const unsigned long long slot = table_find<KEYW>(d, key, true);
    *val_ptr<VALW>(d, slot) = val_pack<VALW>(d, 0u, (unsigned)parenti);
    bucket_push(d, f, (uint32_t)slot);
    d.ctrl->inserted = 1;
    d.ctrl->pushed = 1;
}

// Walk parenti from the final coordinate to the origin (backtrace.cpp:44-69); one thread.
template <int KEYW, int VALW>
__global__ void backtrace_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevSearch d, uint32_t *out, int max_cols)
{
    int pos[PG_MAX_SEQ];
    for (int i = 0; i < p.n; i++) pos[i] = p.len[i];
    int cols = 0;
    int g_final = -1;
    for (;;) {
        bool origin = true;
        Key<KEYW> key = Key<KEYW>::zero();
        for (int i = 0; i < p.n; i++) {
            if (pos[i]) origin = false;
            key.add_val((unsigned)pos[i], i * p.key_bits);
        }
        if (origin || cols >= max_cols) break;
        const unsigned long long slot = table_find<KEYW>(d, key, false); // read-only probe
        const typename ValT<VALW>::T val = slot == ~0ull ? 0 : *val_ptr<VALW>(d, slot);
        if (val == 0) {
            out[0] = 0xffffffffu;
            return;
        }
        if (cols == 0) g_final = (int)val_g<VALW>(d, val);
        const unsigned mask = val_mask<VALW>(d, val);
        out[2 + cols] = mask;
        cols++;
        for (int i = 0; i < p.n; i++) pos[i] -= (mask >> i) & 1;
    }
    out[0] = (uint32_t)cols;
    out[1] = (uint32_t)g_final;
}

// Host-side table lookup of one coordinate (distributed backtrace).
template <int KEYW, int VALW>
__global__ void lookup_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevSearch d, const uint16_t *pos, int *out)
{
    Key<KEYW> key = Key<KEYW>::zero();
    for (int i = 0; i < p.n; i++) key.add_val((unsigned)pos[i], i * p.key_bits);
    out[0] = 0;
    const unsigned long long slot = table_find<KEYW>(d, key, false);
    if (slot == ~0ull) return;
    const typename ValT<VALW>::T val = *val_ptr<VALW>(d, slot);
    if (val == 0) return;
    out[0] = 1;
    out[1] = (int)val_g<VALW>(d, val);
    out[2] = (int)val_mask<VALW>(d, val);
    out[3] = val_closed<VALW>(d, val) ? 0 : 1;
}

// The same lookup for many coordinates, one thread each: state 0 absent / 1 open / 2 closed, g and move mask (-1 when
// absent).  Read-only, so it may run between rounds; table checks look up whole lattices or frontiers through it.
template <int KEYW, int VALW>
__global__ void lookup_batch_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevSearch d, const uint16_t *pos,
                                    long long count, int *state, int *g, int *parenti)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        Key<KEYW> key = Key<KEYW>::zero();
        for (int k = 0; k < p.n; k++) key.add_val((unsigned)pos[i * p.n + k], k * p.key_bits);
        int st = 0, gv = -1, pm = -1;
        const unsigned long long slot = table_find<KEYW>(d, key, false);
        if (slot != ~0ull) {
            const typename ValT<VALW>::T val = *val_ptr<VALW>(d, slot);
            if (val != 0) {
                st = val_closed<VALW>(d, val) ? 2 : 1;
                gv = (int)val_g<VALW>(d, val);
                pm = (int)val_mask<VALW>(d, val);
            }
        }
        state[i] = st;
        g[i] = gv;
        parenti[i] = pm;
    }
}

// Count open / closed entries at the end (PAStar.cpp:591-619 report): every value of every block in use.  out[0] / out[1]
// count open / closed entries; out[2] (set to LLONG_MAX by the caller) receives the min of g + h (unweighted h) over the open
// entries, the open-list part of the search's lower bound: the coordinate is decoded from the block's directory key and
// the value's place in the block, and h gathered from the P pair tables.
template <int KEYW, int VALW>
__global__ void census_kernel(const __grid_constant__ DevProblem p, const __grid_constant__ DevSearch d, unsigned long long *out)
{
    unsigned long long open = 0, closed = 0;
    long long lb = LLONG_MAX;
    const unsigned long long nvals = (d.dir_mask + 1) << d.D;
    const unsigned fmask = (1u << p.key_bits) - 1u;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < nvals; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long *e = d.dir + (i >> d.D) * KEYW;
        const bool used = KEYW == 1 ? e[0] != 0 : (e[0] != 0 || e[1] != 0);
        if (!used) continue;
        const typename ValT<VALW>::T val = *val_ptr<VALW>(d, i);
        if (val == 0) continue;
        if (val_closed<VALW>(d, val)) {
            closed++;
            continue;
        }
        open++;
        Key<KEYW> bkey;
        bkey.lo = KEYW == 1 ? e[0] - 1 : e[0];
        if constexpr (KEYW == 2) bkey.hi = e[1] & ~(1ull << 63);
        const Key<KEYW> key = block_entry_key<KEYW>(d, bkey, (unsigned)(i & ((1ull << d.D) - 1)));
        long long h = 0;
        for (int pr = 0; pr < p.npairs; pr++)
            h += (long long)pg_table_cell(p, pr, (int)key.field(p.pa[pr] * p.key_bits, fmask), (int)key.field(p.pb[pr] * p.key_bits, fmask)) * p.w[pr];
        lb = min(lb, (long long)val_g<VALW>(d, val) + h);
    }
    for (int o = 16; o; o >>= 1) {
        open += __shfl_down_sync(0xffffffffu, open, o);
        closed += __shfl_down_sync(0xffffffffu, closed, o);
        lb = min(lb, __shfl_down_sync(0xffffffffu, lb, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (open) atomicAdd(out, open);
        if (closed) atomicAdd(out + 1, closed);
        if (lb != LLONG_MAX) atomicMin(reinterpret_cast<long long *>(out + 2), lb);
    }
}

__global__ void fill_u64_kernel(unsigned long long *p, unsigned long long v, long long n)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}

// run STMT with KW / VW bound to the table's key width (u64 words) and value width (bytes): (1,4), (1,8) or (2,8)
#define PG_DISPATCH_KV(s, STMT)                  \
    do {                                         \
        if ((s)->keyw == 1 && (s)->valw == 4) {  \
            constexpr int KW = 1, VW = 4;        \
            STMT;                                \
        } else if ((s)->keyw == 1) {             \
            constexpr int KW = 1, VW = 8;        \
            STMT;                                \
        } else {                                 \
            constexpr int KW = 2, VW = 8;        \
            STMT;                                \
        }                                        \
    } while (0)

int ilog2i(int v)
{
    int l = 0;
    while ((1 << (l + 1)) <= v) l++;
    return l;
}

DevSearch dev_search(const pg_ctx *ctx)
{
    const SearchState *s = ctx->search;
    DevSearch d;
    d.dir = s->d_dir;
    d.dir_mask = s->dir_slots - 1;
    d.vals = s->d_vals;
    d.kb = ctx->dp.key_bits;
    d.D = s->D;
    d.DL = s->DL;
    d.nb = s->nb;
    d.gs = s->gs;
    {
        int lines_lg = 0;
        while ((1ull << (lines_lg + 1)) <= (s->dir_slots >> (s->keyw == 1 ? 4 : 3))) lines_lg++;
        d.hshift = 32 - std::min(lines_lg, 32); // dir_slots <= 2^25: at most 2^22 lines
    }
    {
        unsigned __int128 low = 0, line = 0;
        for (int i = 0; i < s->D; i++) low |= (unsigned __int128)1 << (i * ctx->dp.key_bits);
        line = low;
        for (int i = 0; i < s->DL; i++) line |= (unsigned __int128)1 << (i * ctx->dp.key_bits + 1);
        d.low_lo = (unsigned long long)low;
        d.low_hi = (unsigned long long)(low >> 64);
        d.line_lo = (unsigned long long)line;
        d.line_hi = (unsigned long long)(line >> 64);
    }
    d.buckets = s->d_buckets;
    d.tail = s->d_tail;
    d.hint = s->d_hint;
    d.pool = s->d_pool;
    d.link = s->d_link;
    d.free_stack = s->d_free;
    for (int i = 0; i < 16; i++) d.free_off[i] = s->free_off[i];
    d.n_units = s->n_units;
    {   // packed key of the final coordinate (Sequences::get_final_coord, Sequences.cpp:53-60)
        unsigned __int128 k = 0;
        for (int i = 0; i < ctx->n; i++) k += (unsigned __int128)(unsigned)ctx->len[i] << (i * ctx->dp.key_bits);
        d.goal_lo = (unsigned long long)k;
        d.goal_hi = (unsigned long long)(k >> 64);
    }
    d.plan = s->d_plan;
    d.plan_cap = s->plan_cap;
    d.ctrl = s->d_ctrl;
    d.n_parts = s->cfg.n_parts;
    d.part = s->cfg.part;
    d.outbox = s->d_outbox;
    d.outbox_count = s->d_outbox_count;
    d.outbox_cap = s->outbox_cap;
    d.p2p = s->p2p ? 1 : 0;
    // P2P mode: this round's half of the double-buffered inboxes / count arrays
    const size_t half = (size_t)s->cfg.n_parts * s->region_bytes;
    for (int i = 0; i < 16; i++) {
        d.peer_inbox[i] = s->peer_inbox[i] ? (char *)s->peer_inbox[i] + (size_t)s->p2p_buf * half : nullptr;
        d.peer_counts[i] = s->peer_counts[i] ? s->peer_counts[i] + (size_t)s->p2p_buf * s->cfg.n_parts : nullptr;
    }
    d.live = s->d_live;
    d.f0 = s->f0;
    d.f_range = s->f_range;
    d.hnum = ctx->wnum;
    d.hsh = ctx->wsh;
    d.hrecip = ctx->wnum > 1 ? (unsigned)((1ull << (32 + ctx->wsh)) / (unsigned long long)ctx->wnum) : 0u; // floor(2^32 / weight) < 2^32
    d.goal_limit = s->goal_limit;
    d.inc_limit = (int)std::min<long long>(s->inc, INT_MAX);
    d.live_cap = s->live_cap;
    d.surv = s->d_surv;
    d.surv_cap = s->surv_cap;
    {
        const int A = ctx->n <= 6 ? 3 : (ctx->n <= 9 ? 4 : 5), HB = ctx->n - A; // ExpCfg<N>
        for (int hi = 0; hi < 16; hi++) {
            unsigned __int128 k = 0;
            if (s->keyw == 1 && HB <= 4)
                for (int b = 0; b < HB; b++)
                    if ((hi >> b) & 1) k += (unsigned __int128)1 << ((A + b) * ctx->dp.key_bits);
            d.keyhigh[hi] = (unsigned long long)k;
        }
    }
    return d;
}

OwnerArgs owner_args(const pg_ctx *ctx)
{
    const SearchState *s = ctx->search;
    OwnerArgs oa;
    memset(&oa, 0, sizeof(oa));
    oa.type = ctx->dp.hash_type;
    oa.shift = ctx->dp.hash_shift;
    const int nd = ctx->dp.hash_type == PG_HASH_PZORDER ? 2 : ctx->n;
    oa.nb = std::min(8, ilog2i(std::max(1, s->cfg.n_parts)) + 2);
    for (int m = 0; m < 8; m++) {
        const int q = ctx->dp.hash_shift + m;
        const int coord = q % nd, bit = q / nd;
        oa.co[m] = bit < ctx->dp.key_bits ? coord : -1;
        oa.bit[m] = bit;
    }
    for (int m = 0; m < oa.nb; m++) { // group the owner-word bits by the coordinate they read
        if (oa.co[m] < 0) continue;
        int k = 0;
        while (k < oa.nfc && oa.fc[k] != oa.co[m]) k++;
        if (k == oa.nfc) oa.fc[oa.nfc++] = oa.co[m];
        oa.fcm[k] |= 1 << m;
    }
    return oa;
}

// MODE as in expand_probe_kernel; inbox = false: this partition's own live parents, true: the parents forwarded by the
// other partitions (MODE 2)
template <int N, int KEYW, int VALW, int MODE, bool LOOPOWN = true>
int launch_expand_round(pg_ctx *ctx, cudaStream_t st, bool inbox)
{
    using C = ExpCfg<N>;
    SearchState *s = ctx->search;
    constexpr int GROUPS = 256 / C::LP;
    constexpr int XW = KEYW == 1 ? 3 : 4;
    constexpr int NI = 1 << C::IB;
#ifdef PG_PFMAX
    constexpr int PFMAX = PG_PFMAX;
#else
    constexpr int PFMAX = (KEYW == 1 && N < 14) ? 8 : 4;
#endif
    constexpr int PF = NI < PFMAX ? NI : PFMAX; // as in the kernel
    const size_t smem = ((sizeof(PairMeta) + 15) & ~size_t(15)) + sizeof(Key<KEYW>) * C::H +
                        sizeof(int) * (size_t)GROUPS * C::GROUP_INTS + (size_t)PF * 256 * (VALW + 12)
#ifdef PG_EXTRA_SMEM
                        + PG_EXTRA_SMEM
#endif
                        ;
    // per-device state (cudaFuncSetAttribute applies to the current device only): cached per context and kernel mode
    int &occ = ctx->occ_expand_probe[MODE == 2 && !LOOPOWN ? 3 : MODE];
    if (!occ) {
        PG_CUDA(ctx, cudaFuncSetAttribute(expand_probe_kernel<N, KEYW, VALW, MODE, LOOPOWN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PG_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, expand_probe_kernel<N, KEYW, VALW, MODE, LOOPOWN>, 256, smem));
        if (occ < 1) occ = 1;
    }
    // persistent grid: resident CTAs per SM x SM count, capped by the parent groups of a full batch
    long long grid = (long long)ctx->sm_count * occ;
    const long long want = (s->batch_target + GROUPS - 1) / GROUPS;
    if (grid > want) grid = std::max<long long>(1, want);
    const DevSearch d = dev_search(ctx);
    ParentSrc ps;
    memset(&ps, 0, sizeof(ps));
    ps.cap = s->live_cap; // == outbox_cap in forwarding mode: the regions of one launch share a layout
    if (!inbox || s->merge_expand) { // this partition's own live parents
        ps.base[ps.n] = s->d_live;
        ps.count[ps.n] = &s->d_ctrl->live_n;
        ps.own |= 1u << ps.n;
        ps.n++;
    }
    if (inbox) { // the parents the other partitions forwarded
        ps.cap = s->outbox_cap;
        for (int src = 0; src < s->cfg.n_parts; src++) {
            if (src == s->cfg.part) continue;
            ps.base[ps.n] = reinterpret_cast<const unsigned long long *>(d.peer_inbox[s->cfg.part]) + (size_t)src * s->outbox_cap * (KEYW + 1);
            ps.count[ps.n] = d.peer_counts[s->cfg.part] + src;
            ps.n++;
        }
    }
    expand_probe_kernel<N, KEYW, VALW, MODE, LOOPOWN><<<(unsigned)grid, 256, smem, st>>>(ctx->dp, d, owner_args(ctx), ps);
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

// does the owner hash read a coordinate that the expand kernel enumerates in its per-lane loop (coordinates >= A)?
template <int N>
bool loop_owner(const pg_ctx *ctx)
{
    using C = ExpCfg<N>;
    const OwnerArgs oa = owner_args(ctx);
    if (oa.type == PG_HASH_PSUM) return false;         // coordinates 0 and 1: lane bits for every N >= 3
    if (oa.type == PG_HASH_FSUM) return N > C::A;
    for (int m = 0; m < oa.nb; m++)
        if (oa.co[m] >= C::A) return true;
    return false;
}

template <int KEYW, int VALW>
int launch_expand_round_k(pg_ctx *ctx, cudaStream_t st, bool inbox = false)
{
    const SearchState *s = ctx->search;
    const int mode = s->cfg.n_parts == 1 ? 0 : (s->forward ? 2 : 1);
    switch (ctx->n) {
#define CASE(X)                                                                    \
    case X:                                                                        \
        if (mode == 0) return launch_expand_round<X, KEYW, VALW, 0>(ctx, st, inbox);     \
        if (mode == 1) return launch_expand_round<X, KEYW, VALW, 1>(ctx, st, inbox);     \
        if (!loop_owner<X>(ctx)) return launch_expand_round<X, KEYW, VALW, 2, false>(ctx, st, inbox); \
        return launch_expand_round<X, KEYW, VALW, 2>(ctx, st, inbox);
#ifdef PG_DEV_BUILD // experiment builds (PG_VARIANT=...): only the sizes the measurements use, a third of the compile time
        CASE(5) CASE(7)
#else
        CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(14) CASE(16)
#define CASE1(X) /* pg_allow_extended_n: the one-partition kernel only */ \
    case X:                                                               \
        if (mode == 0) return launch_expand_round<X, KEYW, VALW, 0>(ctx, st, inbox); \
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, "the partitioned search is not built for this number of sequences");
        CASE1(11) CASE1(12) CASE1(13) CASE1(15)
#undef CASE1
#endif
#undef CASE
    }
    return pg_fail(ctx, PG_ERR_ARG, "unsupported number of sequences");
}

int prof_event(pg_ctx *ctx)
{
    SearchState *s = ctx->search;
    if (s->prof_used == s->prof_ev.size()) {
        cudaEvent_t e;
        PG_CUDA(ctx, cudaEventCreate(&e));
        s->prof_ev.push_back(e);
    }
    PG_CUDA(ctx, cudaEventRecord(s->prof_ev[s->prof_used++], ctx->stream));
    return PG_OK;
}

constexpr size_t PROF_PER_ROUND = 5; // before select, claim, expand, insert, after insert

int prof_harvest(pg_ctx *ctx) // after a stream synchronise
{
    SearchState *s = ctx->search;
    for (size_t i = 0; i + PROF_PER_ROUND <= s->prof_used; i += PROF_PER_ROUND) {
        float t[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; k++) PG_CUDA(ctx, cudaEventElapsedTime(&t[k], s->prof_ev[i + k], s->prof_ev[i + k + 1]));
        s->select_ms += t[0];
        s->claim_ms += t[1];
        s->expand_ms += t[2];
        s->insert_ms += t[3];
    }
    s->prof_used = 0;
    for (size_t i = 0; i + 2 <= s->prof_used2; i += 2) {
        float t = 0;
        PG_CUDA(ctx, cudaEventElapsedTime(&t, s->prof_ev2[i], s->prof_ev2[i + 1]));
        s->inbox_ms += t;
    }
    s->prof_used2 = 0;
    return PG_OK;
}

int prof_event2(pg_ctx *ctx)
{
    SearchState *s = ctx->search;
    if (s->prof_used2 == s->prof_ev2.size()) {
        cudaEvent_t e;
        PG_CUDA(ctx, cudaEventCreate(&e));
        s->prof_ev2.push_back(e);
    }
    PG_CUDA(ctx, cudaEventRecord(s->prof_ev2[s->prof_used2++], ctx->stream));
    return PG_OK;
}

// records at `recs`, their count in device memory at n_ptr (at most n_max)
int launch_insert(pg_ctx *ctx, const void *recs, const unsigned long long *n_ptr, unsigned long long n_max)
{
    SearchState *s = ctx->search;
    if (n_max == 0) return PG_OK;
    const long long grid = std::min<long long>((long long)((n_max + 1023) / 1024), (long long)ctx->sm_count * 2 * PG_INS_CTAS);
    PG_DISPATCH_KV(s, (insert_kernel<KW, VW><<<(unsigned)grid, 256, 0, ctx->stream>>>(dev_search(ctx), (const unsigned long long *)recs, n_ptr, n_max)));
    PG_CUDA(ctx, cudaGetLastError());
    return PG_OK;
}

// host-known counts go through a small device array (pinned staging is overkill: 64 values, once per call)
int launch_insert_host_count(pg_ctx *ctx, const void *recs, unsigned long long n, int which)
{
    SearchState *s = ctx->search;
    if (n == 0) return PG_OK;
    unsigned long long *slot = s->d_host_counts + which;
    PG_CUDA(ctx, cudaMemcpyAsync(slot, &s->h_host_counts[which], 8, cudaMemcpyHostToDevice, ctx->stream));
    return launch_insert(ctx, recs, slot, n);
}

int launch_round(pg_ctx *ctx, int f_limit)
{
    SearchState *s = ctx->search;
    int rc;
    if (s->profile && (rc = prof_event(ctx)) != PG_OK) return rc;
    select_kernel<<<1, SELECT_THREADS, 0, ctx->stream>>>(dev_search(ctx), (long long)s->batch_target, f_limit);
    PG_CUDA(ctx, cudaGetLastError());
    if (s->profile && (rc = prof_event(ctx)) != PG_OK) return rc;
    {
        const long long grid = std::min<long long>((s->batch_target + 256 * PG_CLAIM_PF - 1) / (256 * PG_CLAIM_PF), (long long)ctx->sm_count * 32); // claim: PG_CLAIM_PF pops per thread
        const long long fgrid = std::min<long long>((s->batch_target + 255) / 256, (long long)ctx->sm_count * 8);
        const DevSearch d = dev_search(ctx);
        PG_DISPATCH_KV(s, (claim_kernel<KW, VW><<<(unsigned)grid, 256, 0, ctx->stream>>>(d)));
        PG_CUDA(ctx, cudaGetLastError());
        if (s->forward) { // the parents and their counts leave at once: they travel while this partition expands its own
            const OwnerArgs oa = owner_args(ctx);
            if (s->keyw == 1)
                forward_kernel<1><<<(unsigned)fgrid, 256, 0, ctx->stream>>>(ctx->dp, d, oa);
            else
                forward_kernel<2><<<(unsigned)fgrid, 256, 0, ctx->stream>>>(ctx->dp, d, oa);
            PG_CUDA(ctx, cudaGetLastError());
            publish_counts_kernel<<<1, 64, 0, ctx->stream>>>(d, s->stamped ? 1 : 0);
            PG_CUDA(ctx, cudaGetLastError());
        }
    }
    if (s->profile && (rc = prof_event(ctx)) != PG_OK) return rc;
    if (!s->merge_expand) {
        PG_DISPATCH_KV(s, (rc = launch_expand_round_k<KW, VW>(ctx, ctx->stream)));
        if (rc != PG_OK) return rc;
    }
    if (s->profile && (rc = prof_event(ctx)) != PG_OK) return rc;
    if (!s->forward) { // forwarding: the survivors are inserted after the forwarded parents have been expanded as well
        if ((rc = launch_insert(ctx, s->d_surv, &s->d_ctrl->surv_n, s->surv_cap)) != PG_OK) return rc;
    }
    if (s->profile && (rc = prof_event(ctx)) != PG_OK) return rc;
    if (!s->forward && s->p2p && s->peer_counts[0]) {
        publish_counts_kernel<<<1, 64, 0, ctx->stream>>>(dev_search(ctx), s->stamped ? 1 : 0);
        PG_CUDA(ctx, cudaGetLastError());
    }
    s->rounds++;
    return PG_OK;
}

} // namespace

int sync_ctrl(pg_ctx *ctx)
{
    SearchState *s = ctx->search;
    PG_CUDA(ctx, cudaMemcpyAsync(s->h_ctrl, s->d_ctrl, sizeof(SearchCtrl), cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (s->profile) {
        int rc = prof_harvest(ctx);
        if (rc != PG_OK) return rc;
    }
    switch (s->h_ctrl->error) {
    case 0:
        return PG_OK;
    case 1:
        return pg_fail(ctx, PG_ERR_CAPACITY, "closed/open hash table is full: raise pg_search_config.table_capacity");
    case 2:
        return pg_fail(ctx, PG_ERR_CAPACITY, "open-list chunk pool exhausted: raise pg_search_config.table_capacity");
    case 3:
        return pg_fail(ctx, PG_ERR_CAPACITY, "f exceeded the bucket range");
    case 5:
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, "a successor's f fell below h(start): the heuristic is not consistent for this cost model");
    case 6:
        return pg_fail(ctx, PG_ERR_STATE, "a peer partition did not deliver its counts for this round (device-side wait timed out)");
    default:
        return pg_fail(ctx, PG_ERR_CAPACITY, "outbox overflow: lower batch_target");
    }
}

void fill_counters(const SearchState *s, pg_result *r)
{
    const SearchCtrl *c = s->h_ctrl;
    r->pops = (int64_t)c->pops;
    r->expansions = (int64_t)c->expansions;
    r->generated = (int64_t)c->generated;
    r->reopen = (int64_t)c->reopen;
    r->rounds = s->rounds;
    r->probed = (int64_t)(c->generated - c->pruned);
    r->pushed = (int64_t)c->pushed;
    r->inserted = (int64_t)c->inserted;
    r->kernel_ms = s->kernel_ms;
    r->expand_ms = s->expand_ms;
    r->select_ms = s->select_ms;
    r->survivors = (int64_t)c->table_used;
    r->inbox_ms = s->inbox_ms;
    r->claim_ms = s->claim_ms;
    r->insert_ms = s->insert_ms;
#ifdef PG_PHASE_TIMING
    fprintf(stderr, "expand phase warp-cycles: prepare %llu pass1 %llu pass2 %llu tail %llu\n", c->phase[2], c->phase[3], c->phase[4], c->phase[5]);
#endif
}

// ---- the large device buffers of a search (value blocks, directory, open-list pool, survivor list: tens of GB) are kept
// for the life of the process and handed to the next search that asks for the same size on the same device: a
// cudaMalloc + cudaFree of 16 GiB costs tens of milliseconds (more when eight processes do it at once), which is most
// of what a sub-second job spends outside its kernels.  pg_release_cached_memory() gives everything back.
namespace {
constexpr size_t BIG_MIN = 64ull << 20;      // smaller buffers go straight to cudaMalloc / cudaFree
constexpr size_t BIG_HELD_MAX = 64ull << 30; // per process; beyond it freed buffers are released
struct BigCache {
    std::mutex m;
    std::multimap<std::pair<int, size_t>, void *> free_list;
    size_t held = 0;
} g_big;

void big_release_all()
{
    std::lock_guard<std::mutex> lk(g_big.m);
    int cur = 0;
    cudaGetDevice(&cur);
    for (auto &kv : g_big.free_list) {
        cudaSetDevice(kv.first.first);
        cudaFree(kv.second);
    }
    g_big.free_list.clear();
    g_big.held = 0;
    cudaSetDevice(cur);
}

cudaError_t big_alloc(int device, void **p, size_t bytes)
{
    if (bytes >= BIG_MIN) {
        std::lock_guard<std::mutex> lk(g_big.m);
        auto it = g_big.free_list.find({device, bytes});
        if (it != g_big.free_list.end()) {
            *p = it->second;
            g_big.held -= bytes;
            g_big.free_list.erase(it);
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMalloc(p, bytes);
    bool held = false;
    if (e == cudaErrorMemoryAllocation) {
        std::lock_guard<std::mutex> lk(g_big.m);
        held = g_big.held != 0;
    }
    if (held) { // make room and try once more
        cudaGetLastError();
        big_release_all();
        e = cudaMalloc(p, bytes);
    }
    return e;
}

// the caller has synchronised the stream(s) that used the buffer
void big_free(int device, void *p, size_t bytes)
{
    if (!p) return;
    if (bytes >= BIG_MIN) {
        std::lock_guard<std::mutex> lk(g_big.m);
        if (g_big.held + bytes <= BIG_HELD_MAX) {
            g_big.free_list.insert({{device, bytes}, p});
            g_big.held += bytes;
            return;
        }
    }
    cudaFree(p);
}
} // namespace

extern "C" void pg_release_cached_memory(void) { big_release_all(); }

void pg_search_free(pg_ctx *ctx)
{
    SearchState *s = ctx->search;
    if (!s) return;
    cudaStreamSynchronize(ctx->stream); // nothing of this search is in flight when its buffers change hands
    big_free(ctx->device, s->d_dir, s->bytes_dir);
    big_free(ctx->device, s->d_vals, s->bytes_vals);
    cudaFree(s->d_buckets);
    cudaFree(s->d_tail);
    cudaFree(s->d_hint);
    big_free(ctx->device, s->d_pool, s->bytes_pool);
    big_free(ctx->device, s->d_link, s->bytes_link);
    cudaFree(s->d_free);
    cudaFree(s->d_plan);
    cudaFree(s->d_ctrl);
    cudaFree(s->d_trace);
    cudaFree(s->d_outbox);
    cudaFree(s->d_outbox_count);
    big_free(ctx->device, s->d_live, s->bytes_live);
    big_free(ctx->device, s->d_surv, s->bytes_surv);
    cudaFree(s->d_host_counts);
    if (s->h_ctrl) cudaFreeHost(s->h_ctrl);
    if (s->h_outbox_count) cudaFreeHost(s->h_outbox_count);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    for (cudaEvent_t e : s->prof_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : s->prof_ev2) cudaEventDestroy(e);
    delete s;
    ctx->search = nullptr;
}

extern "C" int pg_xrec_stride(const pg_ctx *ctx)
{
    if (!ctx) return 0;
    return ctx->n * ctx->dp.key_bits <= 63 ? 24 : 32;
}

extern "C" int pg_search_begin(pg_ctx *ctx, const pg_search_config *cfg)
{
    if (!ctx || !cfg || cfg->n_parts < 1 || cfg->n_parts > 64 || cfg->part < 0 || cfg->part >= cfg->n_parts) return PG_ERR_ARG;
    if (!ctx->tables_built) return pg_fail(ctx, PG_ERR_STATE, "pg_build_pair_tables has not run");
    if (cfg->n_parts > 1 && (ctx->n == 11 || ctx->n == 12 || ctx->n == 13 || ctx->n == 15))
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, "the partitioned search is not built for this number of sequences (pg_allow_extended_n: one GPU only)");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    pg_search_free(ctx);
    SearchState *s = new SearchState();
    ctx->search = s;
    ctx->lb_valid = false;
    s->cfg = *cfg;
    s->keyw = ctx->n * ctx->dp.key_bits <= 63 ? 1 : 2;
    if (s->keyw == 2 && ctx->n * ctx->dp.key_bits > 127) return pg_fail(ctx, PG_ERR_UNSUPPORTED, "packed coordinate key exceeds 127 bits");
    s->xrec = pg_xrec_stride(ctx);
    s->D = std::min(ctx->n, 7);
    s->DL = ctx->dp.key_bits >= 2 ? std::min(ctx->n, s->keyw == 1 ? 4 : 3) : 0;
    ctx->occ_expand_probe[0] = ctx->occ_expand_probe[1] = ctx->occ_expand_probe[2] = ctx->occ_expand_probe[3] = 0; // the value width may differ from the last search's

    s->batch_target = cfg->batch_target > 0 ? cfg->batch_target : 16384;

    // ---- f range: [h(start), cost of the all-advance path]
    int *d_tmp;
    PG_CUDA(ctx, cudaMalloc(&d_tmp, 64));
    std::vector<uint16_t> zero(ctx->n, 0);
    uint16_t *d_zero;
    PG_CUDA(ctx, cudaMalloc(&d_zero, 64));
    PG_CUDA(ctx, cudaMemcpy(d_zero, zero.data(), ctx->n * 2, cudaMemcpyHostToDevice));
    int rc = pg_launch_calc_h(ctx, d_zero, 1, d_tmp, ctx->stream);
    if (rc != PG_OK) return rc;
    PG_CUDA(ctx, cudaMemcpyAsync(&s->f0, d_tmp, 4, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(d_tmp);
    cudaFree(d_zero);
    {   // the all-advance path (column t moves every sequence with t < len) is an alignment: an upper bound on g*
        std::vector<uint32_t> advance;
        for (int t = 0;; t++) {
            uint32_t m = 0;
            for (int i = 0; i < ctx->n; i++) m |= (uint32_t)(t < ctx->len[i]) << i;
            if (!m) break;
            advance.push_back(m);
        }
        s->ub = (int)std::min<long long>(pg_path_cost(ctx, advance), INT_MAX - 1);
    }
    // weighted search: a kept successor has g <= UB and f_w <= floor(weight * UB); the floor stays h(start) <= g + h <= f_w
    const long long wub = ((long long)s->ub * ctx->wnum) >> ctx->wsh;
    if (wub >= INT_MAX)
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, "weight x upper bound does not fit 32 bits");
    // incumbent of cost U: only what can beat U is kept - exact: f < U; weighted: g < U, f_w <= floor(weight * U) - so the
    // bucket range, the prune and goal limits and the value width shrink with U.  They carry the whole bound of the exact
    // search; the weighted one also drops successors by their lower bound (DevSearch::inc_limit).
    s->inc = ctx->inc_cost >= 0 ? ctx->inc_cost : LLONG_MAX;
    const long long winc = s->inc == LLONG_MAX ? LLONG_MAX : (s->inc * ctx->wnum) >> ctx->wsh;
    const long long f_end = std::min(wub, winc);                                 // last bucket's f
    const long long f_lim = ctx->wnum > 1 ? f_end + 1 : std::min(wub + 1, s->inc); // successors with f >= this are dropped
    long long range = f_end - s->f0 + 2;
    if (range < 2) range = 2;
    if (range > (1ll << 27)) // 1 GiB of bucket heads at most: a wider f range is refused, never clamped
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, "f range (weight x upper bound - h(start)) exceeds 2^27 open-list buckets");
    s->f_range = (int)range;
    s->goal_limit = (int)std::min(std::min((long long)s->ub + 1, s->inc), (long long)s->f0 + s->f_range);

    // ---- value width: 4 bytes when g (<= the upper bound), the open bit and the move mask fit 32 bits
    {
        const char *fv = getenv("PG_VALW"); // PG_VALW=8 forces the wide form (tests)
        const bool fits = s->keyw == 1 && (unsigned long long)std::min((long long)s->ub, s->inc - 1) + 2ull < (1ull << (31 - ctx->n));
        s->valw = (fits && !(fv && atoi(fv) == 8)) ? 4 : 8;
        s->nb = s->valw == 4 ? ctx->n : 31;
        s->gs = s->nb + 1;
    }
    // ---- capacity.  table_capacity counts the coordinates the caller wants room for; blocks are cubes of 2^D
    //      coordinates of which a search fills a part (the frontier's surface cuts through them), so four value slots are
    //      provided per coordinate: 16 B per coordinate with 4-byte values, as much as a keyed 16-byte entry took.
    {
        size_t free_b = 0, total_b = 0;
        PG_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
        const uint64_t per_coord = 4ull * (uint64_t)s->valw + 24; // values + open-list pool share
        uint64_t want = cfg->table_capacity > 0 ? (uint64_t)cfg->table_capacity : 0;
        if (want == 0) {
            want = 1024;
            while (want * 2 * per_coord <= free_b / 2 && want * 2 <= (1ull << 30)) want *= 2; // about half of what is free
            // ... but never more than the lattice itself (small inputs would otherwise spend their run time clearing GBs)
            long double lattice = 1.0L;
            for (int i = 0; i < ctx->n; i++) lattice *= (long double)(ctx->len[i] + 2);
            uint64_t need = 1024;
            while ((long double)need < lattice && need < want) need *= 2;
            want = std::min(want, need);
        }
        uint64_t slots = 1ull << (s->D + 5); // at least two directory lines
        while (slots < 4 * want && slots < (1ull << 32)) slots *= 2; // u32 slot ids in the open buckets
        s->cap = slots;
        s->dir_slots = slots >> s->D;
    }
    const uint64_t cap = std::max<uint64_t>(s->cap / 4, 1024); // coordinates provided for: sizes the open-list pool

    // ---- allocations
    s->bytes_dir = (size_t)s->dir_slots * 8 * s->keyw;
    PG_CUDA(ctx, big_alloc(ctx->device, (void **)&s->d_dir, s->bytes_dir));
    PG_CUDA(ctx, cudaMemsetAsync(s->d_dir, 0, (size_t)s->dir_slots * 8 * s->keyw, ctx->stream));
    s->bytes_vals = (size_t)s->cap * s->valw;
    PG_CUDA(ctx, big_alloc(ctx->device, (void **)&s->d_vals, s->bytes_vals));
    PG_CUDA(ctx, cudaMemsetAsync(s->d_vals, 0, (size_t)s->cap * s->valw, ctx->stream));
    PG_CUDA(ctx, cudaMalloc(&s->d_buckets, (size_t)s->f_range * 8));
    PG_CUDA(ctx, cudaMalloc(&s->d_tail, (size_t)s->f_range * 4));
    PG_CUDA(ctx, cudaMemsetAsync(s->d_tail, 0, (size_t)s->f_range * 4, ctx->stream));
    PG_CUDA(ctx, cudaMalloc(&s->d_hint, (size_t)s->f_range * 4));
    PG_CUDA(ctx, cudaMemsetAsync(s->d_hint, 0, (size_t)s->f_range * 4, ctx->stream));
    fill_u64_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(s->d_buckets, BUCKET_EMPTY, (long long)s->f_range);
    PG_CUDA(ctx, cudaGetLastError());
    // Every table slot is pushed once per improvement.  Chunk sizes double, so a bucket wastes at most its own
    // size; each non-empty bucket holds at least one unit.
    uint64_t units = 5 * (cap / UNIT) + (uint64_t)s->f_range + 4096; // measured: 2.7 pushes per table entry + chunk slack
    s->n_units = (uint32_t)std::min<uint64_t>(units, 0x7ffffff0ull);
    s->bytes_pool = (size_t)s->n_units * UNIT * 4;
    PG_CUDA(ctx, big_alloc(ctx->device, (void **)&s->d_pool, s->bytes_pool));
    s->bytes_link = (size_t)s->n_units * 8;
    PG_CUDA(ctx, big_alloc(ctx->device, (void **)&s->d_link, s->bytes_link));
    {   // free stacks: class lg can never hold more than n_units >> lg chunks
        uint32_t tot = 0;
        for (uint32_t lg = 0; lg <= MAXLG; lg++) {
            s->free_off[lg] = tot;
            tot += (s->n_units >> lg) + 1;
        }
        PG_CUDA(ctx, cudaMalloc(&s->d_free, (size_t)tot * 4));
    }
    // a round pops at most ~2*target entries: the bucket crossing the target may add one chunk of up to the
    // entries already taken.  Plan entries: one per chunk.
    s->plan_cap = (uint32_t)(SELECT_THREADS * (MAXLG + 4) + 64);
    PG_CUDA(ctx, cudaMalloc(&s->d_plan, (size_t)s->plan_cap * sizeof(PlanEntry)));
    PG_CUDA(ctx, cudaMalloc(&s->d_ctrl, sizeof(SearchCtrl)));
    PG_CUDA(ctx, cudaMallocHost(&s->h_ctrl, sizeof(SearchCtrl)));
    {
        size_t total = 0;
        for (int i = 0; i < ctx->n; i++) total += (size_t)ctx->len[i];
        PG_CUDA(ctx, cudaMalloc(&s->d_trace, std::max<size_t>(1u << 16, (total + 64) * 4)));
    }
    PG_CUDA(ctx, cudaEventCreate(&s->ev0));
    PG_CUDA(ctx, cudaEventCreate(&s->ev1));
    {
        // live parents: at most one per popped entry; survivors: at most every successor of every live parent
        const uint64_t S = (1ull << ctx->n) - 1;
        s->live_cap = (uint64_t)s->batch_target + UNIT;
        s->bytes_live = (size_t)s->live_cap * (s->keyw + 1) * 8;
        PG_CUDA(ctx, big_alloc(ctx->device, (void **)&s->d_live, s->bytes_live));
        s->surv_cap = (uint64_t)(s->batch_target + UNIT) * S + 64;
        s->bytes_surv = (size_t)s->surv_cap * s->xrec;
        PG_CUDA(ctx, big_alloc(ctx->device, (void **)&s->d_surv, s->bytes_surv));
        PG_CUDA(ctx, cudaMalloc(&s->d_host_counts, 8 * 64));
    }
    if (cfg->n_parts > 1) {
        s->forward = cfg->reserved == 2;
        s->merge_expand = s->forward && getenv("PG_MERGE_EXPAND") && atoi(getenv("PG_MERGE_EXPAND")) != 0;
        if (s->forward) {
            // parent forwarding: a destination receives at most every live parent of the round
            s->outbox_cap = (uint64_t)s->batch_target + UNIT;
            s->region_bytes = (size_t)s->outbox_cap * (s->keyw + 1) * 8;
        } else {
            // worst case every successor of a full batch goes to one destination
            const uint64_t S = (1ull << ctx->n) - 1;
            s->outbox_cap = (uint64_t)(s->batch_target + UNIT) * S;
            // beyond four partitions the worst case is sized at 4x the share a uniform hash gives one destination; a round
            // that needs more ends the run with PG_ERR_CAPACITY ("outbox overflow") instead of writing out of bounds
            if (cfg->n_parts > 4) s->outbox_cap = s->outbox_cap * 4 / cfg->n_parts;
            s->outbox_cap += (uint64_t)OBOX_CHUNK * 8 * (uint64_t)ctx->sm_count;
            s->region_bytes = (size_t)s->outbox_cap * s->xrec;
            if (cfg->reserved != 1) // reserved == 1: P2P mode, records go straight to the peers' inboxes (pg_search_set_peers)
                PG_CUDA(ctx, cudaMalloc(&s->d_outbox, (size_t)cfg->n_parts * s->outbox_cap * s->xrec));
        }
        PG_CUDA(ctx, cudaMalloc(&s->d_outbox_count, 8 * 64));
        PG_CUDA(ctx, cudaMallocHost(&s->h_outbox_count, 8 * 64));
        PG_CUDA(ctx, cudaMemsetAsync(s->d_outbox_count, 0, 8 * 64, ctx->stream));
    }

    SearchCtrl c;
    memset(&c, 0, sizeof(c));
    c.f0 = s->f0;
    c.f_range = s->f_range;
    c.cursor = 0;
    c.best_goal = INT_MAX;
    c.prune_limit = (int)std::min(f_lim, (long long)s->f0 + s->f_range);
    c.min_open_f = s->f0;
    c.drop_lb = INT_MAX;
    PG_CUDA(ctx, cudaMemcpyAsync(s->d_ctrl, &c, sizeof(c), cudaMemcpyHostToDevice, ctx->stream));
    // PAStar.cpp:153 enqueues the start node on rank 0 / OpenList[0] whatever its owner; here its true owner
    // (get_id of the origin is 0 for every hash) which is partition 0 as well.
    if (cfg->part == 0) {
        const int parenti = (1 << ctx->n) - 1; // Sequences.cpp:75
        PG_DISPATCH_KV(s, (seed_kernel<KW, VW><<<1, 1, 0, ctx->stream>>>(dev_search(ctx), s->f0, parenti)));
        PG_CUDA(ctx, cudaGetLastError());
    }
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    s->active = true;
    return PG_OK;
}

extern "C" int pg_search_round(pg_ctx *ctx, int32_t f_limit)
{
    if (!ctx || !ctx->search || !ctx->search->active) return ctx ? pg_fail(ctx, PG_ERR_STATE, "pg_search_begin has not run") : PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    if (s->cfg.n_parts > 1 && s->cfg.reserved >= 1 && !s->p2p) return pg_fail(ctx, PG_ERR_STATE, "P2P mode requested but pg_search_set_peers has not run");
    int rc = launch_round(ctx, f_limit);
    if (rc != PG_OK) return rc;
    if (s->cfg.n_parts > 1)
        PG_CUDA(ctx, cudaMemcpyAsync(s->h_outbox_count, s->d_outbox_count, 8 * 64, cudaMemcpyDeviceToHost, ctx->stream));
    return sync_ctrl(ctx);
}

extern "C" int pg_search_round_async(pg_ctx *ctx, int32_t f_limit)
{
    if (!ctx || !ctx->search || !ctx->search->active) return ctx ? pg_fail(ctx, PG_ERR_STATE, "pg_search_begin has not run") : PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    if (s->cfg.n_parts > 1 && s->cfg.reserved >= 1 && !s->p2p) return pg_fail(ctx, PG_ERR_STATE, "P2P mode requested but pg_search_set_peers has not run");
    return launch_round(ctx, f_limit);
}

extern "C" int pg_search_sync(pg_ctx *ctx)
{
    if (!ctx || !ctx->search || !ctx->search->active) return ctx ? pg_fail(ctx, PG_ERR_STATE, "pg_search_begin has not run") : PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    return sync_ctrl(ctx);
}

extern "C" int pg_search_rounds(pg_ctx *ctx, int32_t rounds, int32_t f_limit)
{
    if (!ctx || !ctx->search || !ctx->search->active) return ctx ? pg_fail(ctx, PG_ERR_STATE, "pg_search_begin has not run") : PG_ERR_ARG;
    if (ctx->search->cfg.n_parts != 1) return pg_fail(ctx, PG_ERR_ARG, "pg_search_rounds is for a single partition");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    const int rc = pg_run_rounds(ctx, rounds, f_limit, 8, !ctx->search->profile && !getenv("PG_NO_GRAPH"));
    return rc != PG_OK ? rc : sync_ctrl(ctx);
}

extern "C" int pg_search_profile(pg_ctx *ctx, int enable)
{
    if (!ctx || !ctx->search) return ctx ? pg_fail(ctx, PG_ERR_STATE, "pg_search_begin has not run") : PG_ERR_ARG;
    ctx->search->profile = enable != 0;
    return PG_OK;
}

extern "C" int pg_search_note_rounds(pg_ctx *ctx, int64_t delta)
{
    if (!ctx || !ctx->search) return ctx ? pg_fail(ctx, PG_ERR_STATE, "pg_search_begin has not run") : PG_ERR_ARG;
    ctx->search->rounds += delta;
    return PG_OK;
}

extern "C" int pg_search_set_peers(pg_ctx *ctx, void *const *peer_inbox, int n)
{
    if (!ctx || !ctx->search || !peer_inbox) return PG_ERR_ARG;
    SearchState *s = ctx->search;
    if (n != s->cfg.n_parts || n > 16) return pg_fail(ctx, PG_ERR_ARG, "pg_search_set_peers: one inbox base per partition, at most 16");
    for (int i = 0; i < n; i++) s->peer_inbox[i] = peer_inbox[i];
    s->p2p = true;
    return PG_OK;
}

extern "C" int pg_search_set_peer_counts(pg_ctx *ctx, void *const *peer_counts, int n, int nbuf)
{
    if (!ctx || !ctx->search || !peer_counts) return PG_ERR_ARG;
    SearchState *s = ctx->search;
    if (n != s->cfg.n_parts || n > 16 || nbuf < 1 || nbuf > 2) return pg_fail(ctx, PG_ERR_ARG, "pg_search_set_peer_counts: one count array per partition, 1 or 2 buffers");
    for (int i = 0; i < n; i++) s->peer_counts[i] = (unsigned long long *)peer_counts[i];
    s->p2p_nbuf = nbuf;
    s->p2p_buf = 0;
    return PG_OK;
}

extern "C" int pg_search_set_device_sync(pg_ctx *ctx, int enable)
{
    if (!ctx || !ctx->search) return PG_ERR_ARG;
    SearchState *s = ctx->search;
    if (enable && (s->p2p_nbuf != 2 || !s->peer_counts[s->cfg.part]))
        return pg_fail(ctx, PG_ERR_STATE, "pg_search_set_device_sync needs pg_search_set_peer_counts with two buffers");
    s->stamped = enable != 0;
    return PG_OK;
}

extern "C" int pg_search_insert_inbox_async(pg_ctx *ctx)
{
    if (!ctx || !ctx->search) return PG_ERR_ARG;
    SearchState *s = ctx->search;
    if (!s->p2p || !s->peer_counts[s->cfg.part]) return pg_fail(ctx, PG_ERR_STATE, "pg_search_insert_inbox_async needs pg_search_set_peers and pg_search_set_peer_counts");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if (s->stamped) { // data-flow synchronisation: wait on the device for every source's count of this exchange round
        wait_counts_kernel<<<1, 64, 0, ctx->stream>>>(dev_search(ctx));
        PG_CUDA(ctx, cudaGetLastError());
    }
    if (s->profile && (rc = prof_event2(ctx)) != PG_OK) return rc;
    if (s->forward) {
        // expand the parents the other partitions forwarded (only the successors this partition owns), then insert
        // the round's survivors: those of its own parents and of the forwarded ones
        PG_DISPATCH_KV(s, (rc = launch_expand_round_k<KW, VW>(ctx, ctx->stream, true)));
        if (rc != PG_OK) return rc;
        if ((rc = launch_insert(ctx, s->d_surv, &s->d_ctrl->surv_n, s->surv_cap)) != PG_OK) return rc;
    } else {
        const DevSearch d = dev_search(ctx);
        for (int src = 0; src < s->cfg.n_parts; src++) {
            if (src == s->cfg.part) continue;
            rc = launch_insert(ctx, d.peer_inbox[s->cfg.part] + (size_t)src * s->region_bytes, d.peer_counts[s->cfg.part] + src, s->outbox_cap);
            if (rc != PG_OK) return rc;
        }
    }
    if (s->profile && (rc = prof_event2(ctx)) != PG_OK) return rc;
    s->p2p_buf = (s->p2p_buf + 1) % s->p2p_nbuf;
    s->xround++;
    return PG_OK;
}

extern "C" int64_t pg_search_region_bytes(const pg_ctx *ctx)
{
    return ctx && ctx->search ? (int64_t)ctx->search->region_bytes : 0;
}

extern "C" int64_t pg_search_outbox_capacity(const pg_ctx *ctx)
{
    return ctx && ctx->search ? (int64_t)ctx->search->outbox_cap : 0;
}

extern "C" int pg_search_outbox_counts_dev(pg_ctx *ctx, void **d_counts)
{
    if (!ctx || !ctx->search || !d_counts) return PG_ERR_ARG;
    *d_counts = ctx->search->d_outbox_count;
    return PG_OK;
}

extern "C" int pg_search_insert_segments_dev(pg_ctx *ctx, const void *base, int64_t stride_bytes, const int64_t *counts, int n)
{
    if (!ctx || !ctx->search || !base || !counts || n < 0 || n > 64) return PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    for (int i = 0; i < n; i++) {
        if (counts[i] <= 0) continue;
        s->h_host_counts[i] = (unsigned long long)counts[i];
        int rc = launch_insert_host_count(ctx, (const char *)base + (size_t)i * stride_bytes, (unsigned long long)counts[i], i);
        if (rc != PG_OK) return rc;
    }
    return sync_ctrl(ctx);
}

extern "C" int pg_search_outbox(pg_ctx *ctx, int dst, void **d_records, int64_t *count)
{
    if (!ctx || !ctx->search || !d_records || !count) return PG_ERR_ARG;
    SearchState *s = ctx->search;
    if (dst < 0 || dst >= s->cfg.n_parts || s->cfg.n_parts < 2) return PG_ERR_ARG;
    *d_records = s->d_outbox + (size_t)dst * s->outbox_cap * s->xrec;
    *count = (int64_t)s->h_outbox_count[dst];
    return PG_OK;
}

extern "C" int pg_search_insert_dev(pg_ctx *ctx, const void *d_records, int64_t count)
{
    if (!ctx || !ctx->search || count < 0 || (count > 0 && !d_records)) return PG_ERR_ARG;
    if (count == 0) return PG_OK;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    s->h_host_counts[63] = (unsigned long long)count;
    int rc = launch_insert_host_count(ctx, d_records, (unsigned long long)count, 63);
    if (rc != PG_OK) return rc;
    return sync_ctrl(ctx);
}

extern "C" int pg_search_status(pg_ctx *ctx, int32_t *min_open_f, int32_t *best_goal_g, pg_result *counters)
{
    if (!ctx || !ctx->search) return PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    // a select with target 0 pops nothing but refreshes cursor / min_open_f
    select_kernel<<<1, SELECT_THREADS, 0, ctx->stream>>>(dev_search(ctx), 0ll, INT_MIN + 1);
    PG_CUDA(ctx, cudaGetLastError());
    int rc = sync_ctrl(ctx);
    if (rc != PG_OK) return rc;
    if (min_open_f) *min_open_f = s->h_ctrl->min_open_f;
    if (best_goal_g) *best_goal_g = s->h_ctrl->best_goal;
    if (counters) {
        memset(counters, 0, sizeof(*counters));
        fill_counters(s, counters);
    }
    return PG_OK;
}

extern "C" int pg_search_lookup(pg_ctx *ctx, const uint16_t *pos, int32_t *found, int32_t *g, int32_t *parenti)
{
    if (!ctx || !ctx->search || !pos || !found) return PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    uint16_t *d_pos = (uint16_t *)s->d_trace;
    int *d_out = (int *)(s->d_trace + 64);
    PG_CUDA(ctx, cudaMemcpyAsync(d_pos, pos, ctx->n * 2, cudaMemcpyHostToDevice, ctx->stream));
    PG_DISPATCH_KV(s, (lookup_kernel<KW, VW><<<1, 1, 0, ctx->stream>>>(ctx->dp, dev_search(ctx), d_pos, d_out)));
    PG_CUDA(ctx, cudaGetLastError());
    int h[4];
    PG_CUDA(ctx, cudaMemcpyAsync(h, d_out, 16, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *found = h[0];
    if (g) *g = h[1];
    if (parenti) *parenti = h[2];
    return PG_OK;
}

extern "C" int pg_search_lookup_batch(pg_ctx *ctx, const uint16_t *pos, int64_t count, int32_t *state, int32_t *g, int32_t *parenti)
{
    if (!ctx || !ctx->search || count < 0 || (count > 0 && (!pos || !state || !g || !parenti))) return PG_ERR_ARG;
    const int n = ctx->n;
    for (int64_t i = 0; i < count; i++)
        for (int k = 0; k < n; k++)
            if ((int)pos[i * n + k] > ctx->len[k])
                return pg_fail(ctx, PG_ERR_ARG, "pg_search_lookup_batch: coordinate " + std::to_string(i) + " has position " +
                                                    std::to_string(pos[i * n + k]) + " in sequence " + std::to_string(k) +
                                                    ", past its length " + std::to_string(ctx->len[k]));
    if (count == 0) return PG_OK;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    SearchState *s = ctx->search;
    const int64_t chunk = std::min<int64_t>(count, 1 << 22); // bounded scratch: 4 Mi coordinates per launch
    void *buf = nullptr;
    PG_CUDA(ctx, cudaMalloc(&buf, (size_t)chunk * (2 * n + 12)));
    int *d_out = (int *)buf;
    uint16_t *d_pos = (uint16_t *)(d_out + 3 * chunk);
    int rc = PG_OK;
    for (int64_t b = 0; b < count && rc == PG_OK; b += chunk) {
        const int64_t k = std::min(chunk, count - b);
        cudaError_t e = cudaMemcpyAsync(d_pos, pos + b * n, (size_t)k * n * 2, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) {
            const unsigned grid = (unsigned)std::min<int64_t>((k + 255) / 256, (int64_t)ctx->sm_count * 16);
            PG_DISPATCH_KV(s, (lookup_batch_kernel<KW, VW><<<grid, 256, 0, ctx->stream>>>(ctx->dp, dev_search(ctx), d_pos, (long long)k,
                                                                                          d_out, d_out + chunk, d_out + 2 * chunk)));
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(state + b, d_out, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(g + b, d_out + chunk, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(parenti + b, d_out + 2 * chunk, (size_t)k * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = pg_fail(ctx, PG_ERR_CUDA, std::string("pg_search_lookup_batch: ") + cudaGetErrorString(e));
    }
    cudaFree(buf);
    return rc;
}

extern "C" int pg_search_end(pg_ctx *ctx)
{
    if (!ctx) return PG_ERR_ARG;
    cudaSetDevice(ctx->device);
    pg_search_free(ctx);
    return PG_OK;
}

int pg_census(pg_ctx *ctx, int64_t *open_size, int64_t *closed_size, long long *open_lb)
{
    SearchState *s = ctx->search;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    unsigned long long *d_cnt = (unsigned long long *)s->d_trace;
    unsigned long long h[3] = {0, 0, (unsigned long long)LLONG_MAX};
    PG_CUDA(ctx, cudaMemcpyAsync(d_cnt, h, 24, cudaMemcpyHostToDevice, ctx->stream));
    PG_DISPATCH_KV(s, (census_kernel<KW, VW><<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(ctx->dp, dev_search(ctx), d_cnt)));
    PG_CUDA(ctx, cudaGetLastError());
    PG_CUDA(ctx, cudaMemcpyAsync(h, d_cnt, 24, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (open_size) *open_size = (int64_t)h[0];
    if (closed_size) *closed_size = (int64_t)h[1];
    *open_lb = (long long)h[2];
    return PG_OK;
}

int pg_backtrace(pg_ctx *ctx, std::vector<uint32_t> &masks, int *goal_g)
{
    SearchState *s = ctx->search;
    int total = 0;
    for (int i = 0; i < ctx->n; i++) total += ctx->len[i];
    PG_DISPATCH_KV(s, (backtrace_kernel<KW, VW><<<1, 1, 0, ctx->stream>>>(ctx->dp, dev_search(ctx), s->d_trace, total)));
    PG_CUDA(ctx, cudaGetLastError());
    std::vector<uint32_t> tr((size_t)total + 2);
    PG_CUDA(ctx, cudaMemcpyAsync(tr.data(), s->d_trace, tr.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (tr[0] == 0xffffffffu) return pg_fail(ctx, PG_ERR_STATE, "backtrace lost the parent chain");
    const int cols = (int)tr[0];
    masks.resize(cols);
    for (int c = 0; c < cols; c++) masks[c] = tr[2 + (cols - 1 - c)]; // stored goal-first
    *goal_g = (int)tr[1];
    return PG_OK;
}

int pg_capture(pg_ctx *ctx, const std::function<int()> &enqueue, GraphExec *exec)
{
    SearchState *s = ctx->search;
    exec->reset();
    if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        return PG_OK;
    }
    const int64_t rounds = s->rounds;
    const int rc = enqueue();
    s->rounds = rounds;
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
    if (rc != PG_OK || e != cudaSuccess || !graph || cudaGraphInstantiate(&exec->exec, graph, 0) != cudaSuccess) {
        cudaGetLastError();
        exec->exec = nullptr;
    }
    if (graph) cudaGraphDestroy(graph);
    return rc;
}

int pg_run_rounds(pg_ctx *ctx, int n, int f_limit, int group, bool allow_graph)
{
    SearchState *s = ctx->search;
    int r = 0, rc;
    if (allow_graph && n >= group && !s->rounds_no_graph) {
        if (s->rounds_exec && (s->rounds_flimit != f_limit || s->rounds_stream != ctx->stream || s->rounds_group != group))
            s->rounds_exec.reset();
        if (!s->rounds_exec) {
            rc = pg_capture(ctx, [&] {
                int e = PG_OK;
                for (int k = 0; k < group && e == PG_OK; k++) e = launch_round(ctx, f_limit);
                return e;
            }, &s->rounds_exec);
            if (rc != PG_OK) return rc;
            s->rounds_no_graph = !s->rounds_exec;
            s->rounds_group = group;
            s->rounds_flimit = f_limit;
            s->rounds_stream = ctx->stream;
        }
        for (; s->rounds_exec && r + group <= n; r += group) {
            PG_CUDA(ctx, cudaGraphLaunch(s->rounds_exec.exec, ctx->stream));
            s->rounds += group;
        }
    }
    for (; r < n; r++)
        if ((rc = launch_round(ctx, f_limit)) != PG_OK) return rc;
    return PG_OK;
}
