// Successor expansion core shared by the stand-alone getNeigh-batch kernel
// (pg_expand.cu) and the fused search kernel (pg_search.cu).
//
// Reference: Node<N>::getNeigh / pairCost / borderCheck / Node ctor
// (pastar/Node.cpp:205-248, 129-152, 69-77, 32-39), Coord<N>::neigh
// (pastar/Coord.cpp:92-106), HeuristicHPair::calculate_h
// (pastar/HeuristicHPair.cpp:73-86).
//
// The reference evaluates, for each of the 2^N-1 move masks, a sum over all
// P = N(N-1)/2 pairs of pairCost(mask)*w for g and a P-term table gather for
// h: S*P branchy terms and S*P dependent gathers per parent.  Both sums are
// quadratic pseudo-boolean functions of the mask bits whose coefficients
// depend on the parent only, so they are factorised here:
//
//   per pair a 4-entry LUT over (bit_x, bit_y):      4*P table gathers / parent
//       LUTg = {GapGap, gap(y), gap(x), cost(rx,ry)} * w   (Node.cpp:129-152)
//       LUTh = T[px+bx][py+by] * w                         (HeuristicHPair.cpp:82)
//   mask = (high << A) | low;  a group of 2^A lanes shares one parent, lane = low
//       B[low]    = sum over pairs inside low + cross pairs with by = 0
//       E_y[low]  = sum_x (LUT_xy[bx,1] - LUT_xy[bx,0])     one per high sequence y
//       HH[high]  = sum over pairs inside high              shared-memory table
//       value(low, high) = B[low] + HH[high] + sum_{y in high} E_y[low]
//
// so a successor costs two adds and two shared loads per sum instead of P
// terms.  All arithmetic is 32-bit signed integer, as in the reference.
#pragma once
#include "pg_internal.cuh"

template <int N>
struct ExpCfg {
    static constexpr int A = N <= 6 ? 3 : (N <= 9 ? 4 : 5); // mask bits enumerated across lanes
    static constexpr int LP = 1 << A;                       // lanes per parent
    static constexpr int HB = N - A;                        // mask bits enumerated in the per-lane loop
    static constexpr int IB = HB < 4 ? HB : 4;              // ... of which unrolled in registers
    static constexpr int UB = HB - IB;                      // ... and looped
    static constexpr int H = 1 << HB;
    static constexpr int P = N * (N - 1) / 2;
    static constexpr int S = (1 << N) - 1;
    static constexpr int NODE_WORDS = (((2 * N + 3) & ~3) + 12) / 4;
    static constexpr int POS_WORDS = ((2 * N + 3) & ~3) / 4;
    // ints of shared memory per parent group: LUTg, LUTh, HHg, HHh, pos, residues
    static constexpr int GROUP_INTS = 8 * P + 2 * H + 2 * PG_MAX_SEQ;
};

// Per-CTA copy of the pair metadata (avoids divergent constant-bank indexing).
struct PairMeta {
    const void *table[PG_MAX_PAIRS];
    int w[PG_MAX_PAIRS];
    int cols[PG_MAX_PAIRS];
    uint8_t pa[PG_MAX_PAIRS], pb[PG_MAX_PAIRS];
};

__device__ __forceinline__ void pg_load_pair_meta(const DevProblem &p, PairMeta *m)
{
    for (int i = threadIdx.x; i < p.npairs; i += blockDim.x) {
        m->table[i] = p.table[i];
        m->w[i] = p.w[i];
        m->cols[i] = p.cols[i];
        m->pa[i] = p.pa[i];
        m->pb[i] = p.pb[i];
    }
}

// Per-lane result of the factorisation for one parent.
template <int N>
struct ExpLane {
    int Bg, Bh;                                       // B[low] (Bg already includes the parent's g)
    int Eg[ExpCfg<N>::HB > 0 ? ExpCfg<N>::HB : 1];    // E_y[low] per high sequence
    int Eh[ExpCfg<N>::HB > 0 ? ExpCfg<N>::HB : 1];
    int alive;                                        // sequences that can still advance (borderCheck, Node.cpp:69-77)
};

// Stage the LUTs / HH table of one parent in the group's shared memory and compute the lane's B and E terms.
// `sub` is the lane's index in the group and its low mask bits, `gmask` the shfl mask of the group's lanes.
// s_grp points at GROUP_INTS ints of shared memory private to the group.
// Weighted search (hnum > 1): every h term is floor(hnum * T * w / 2^hsh) instead of T * w, so the h sums are
// h_w = sum over pairs of floor(weight * term), with h <= h_w <= weight * h (weight = hnum / 2^hsh >= 1).
template <int N>
__device__ __forceinline__ void pg_expand_prepare(const DevProblem &p, const PairMeta *meta, int *s_grp, const int (&pos)[N], int g,
                                                  int parenti, int sub, unsigned gmask, ExpLane<N> &L, int hnum = 1, int hsh = 0)
{
    using C = ExpCfg<N>;
    int *s_lutg = s_grp;
    int *s_luth = s_grp + 4 * C::P;
    int *s_hhg = s_grp + 8 * C::P;
    int *s_hhh = s_hhg + C::H;
    int *s_pos = s_hhh + C::H; // N positions, then N residues

    int alive = 0;
#pragma unroll
    for (int i = 0; i < N; i++) alive |= (pos[i] < p.len[i]) << i;
    L.alive = alive;
    if (sub < N) {
        int v = 0;
#pragma unroll
        for (int i = 0; i < N; i++)
            if (i == sub) v = pos[i];
        s_pos[sub] = v;
        s_pos[PG_MAX_SEQ + sub] = (int)__ldg(p.seq[sub] + v); // Node.cpp:225 reads seq[len] at the border: padded 0
    }
    __syncwarp(gmask);

    // ---- per-pair LUTs: 4*P entries strided over the group's lanes.  All gathers are issued first (no shared
    //      stores in between), so the L2 latencies of a lane's entries overlap.
    constexpr int NE = (4 * C::P + C::LP - 1) / C::LP;
    int tv[NE], cv[NE];
#pragma unroll
    for (int j = 0; j < NE; j++) {
        const int e = sub + j * C::LP;
        tv[j] = 0;
        cv[j] = 0;
        if (e < 4 * C::P) {
            const int pr = e >> 2, dx = e & 1, dy = (e >> 1) & 1;
            const int x = meta->pa[pr], y = meta->pb[pr];
            // moves that leave the lattice are never emitted; clamp so the gather stays in bounds
            const int ix = min(s_pos[x] + dx, p.len[x]), iy = min(s_pos[y] + dy, p.len[y]);
            const size_t cell = (size_t)ix * meta->cols[pr] + iy;
            tv[j] = p.cell16 ? (int)__ldg(reinterpret_cast<const uint16_t *>(meta->table[pr]) + cell)
                             : __ldg(reinterpret_cast<const int32_t *>(meta->table[pr]) + cell);
            if (dx & dy) cv[j] = __ldg(p.cost + s_pos[PG_MAX_SEQ + x] * 90 + s_pos[PG_MAX_SEQ + y]);
        }
    }
#pragma unroll
    for (int j = 0; j < NE; j++) {
        const int e = sub + j * C::LP;
        if (e < 4 * C::P) {
            const int pr = e >> 2, dx = e & 1, dy = (e >> 1) & 1;
            const int x = meta->pa[pr], y = meta->pb[pr];
            const int w = meta->w[pr];
            // match / mismatch (both move); a gap in the sequence that stays (Node.cpp:140,149-151: opened if that
            // sequence moved into the parent, extended otherwise); gap-gap (Node.cpp:142).  dx and dy are the same for all
            // of a lane's entries (e = sub + j * LP), so this is selects, not branches.
            const int stays = dx ? y : x;
            const int gapc = ((parenti >> stays) & 1) ? p.gap_open : p.gap_ext;
            const int c = (dx & dy) ? cv[j] : ((dx | dy) ? gapc : p.gap_gap);
            s_lutg[e] = c * w;
            s_luth[e] = hnum > 1 ? (int)(((long long)tv[j] * w * hnum) >> hsh) : tv[j] * w;
        }
    }
    __syncwarp(gmask);

    // ---- HH[high]: pairs with both sequences in the high part
    for (int hi = sub; hi < C::H; hi += C::LP) {
        int sg = 0, sh = 0;
#pragma unroll
        for (int y = C::A; y < N; y++) {
#pragma unroll
            for (int z = y + 1; z < N; z++) {
                const int pr = y * N - y * (y + 1) / 2 + (z - y - 1);
                const int idx = pr * 4 + ((hi >> (y - C::A)) & 1) + 2 * ((hi >> (z - C::A)) & 1);
                sg += s_lutg[idx];
                sh += s_luth[idx];
            }
        }
        s_hhg[hi] = sg;
        s_hhh[hi] = sh;
    }

    // ---- B[low], E_y[low]
    int Bg = g, Bh = 0;
#pragma unroll
    for (int x = 0; x < C::A; x++) {
#pragma unroll
        for (int y = x + 1; y < C::A; y++) {
            const int pr = x * N - x * (x + 1) / 2 + (y - x - 1);
            const int idx = pr * 4 + ((sub >> x) & 1) + 2 * ((sub >> y) & 1);
            Bg += s_lutg[idx];
            Bh += s_luth[idx];
        }
    }
#pragma unroll
    for (int y = C::A; y < N; y++) {
        int g0 = 0, g1 = 0, h0 = 0, h1 = 0;
#pragma unroll
        for (int x = 0; x < C::A; x++) {
            const int pr = x * N - x * (x + 1) / 2 + (y - x - 1);
            const int idx = pr * 4 + ((sub >> x) & 1);
            g0 += s_lutg[idx];
            g1 += s_lutg[idx + 2];
            h0 += s_luth[idx];
            h1 += s_luth[idx + 2];
        }
        Bg += g0;
        Bh += h0;
        L.Eg[y - C::A] = g1 - g0;
        L.Eh[y - C::A] = h1 - h0;
    }
    L.Bg = Bg;
    L.Bh = Bh;
    __syncwarp(gmask);
}

// rank of `mask` among the submasks of `alive` in ascending order, minus one (compress mask onto alive's bits)
template <int N>
__device__ __forceinline__ int pg_mask_rank(int mask, int alive)
{
    int r = 0, o = 0;
#pragma unroll
    for (int b = 0; b < N; b++) {
        if ((alive >> b) & 1) {
            r |= ((mask >> b) & 1) << o;
            o++;
        }
    }
    return r - 1;
}

// g / h sums of the 2^IB masks that share the upper high bits `u`, by recursive doubling in registers
template <int N>
__device__ __forceinline__ void pg_expand_block(const ExpLane<N> &L, int u, int (&vg)[1 << ExpCfg<N>::IB], int (&vh)[1 << ExpCfg<N>::IB])
{
    using C = ExpCfg<N>;
    vg[0] = L.Bg;
    vh[0] = L.Bh;
#pragma unroll
    for (int b = 0; b < C::UB; b++) {
        if ((u >> b) & 1) {
            vg[0] += L.Eg[C::IB + b];
            vh[0] += L.Eh[C::IB + b];
        }
    }
#pragma unroll
    for (int b = 0; b < C::IB; b++) {
#pragma unroll
        for (int i = 0; i < (1 << b); i++) {
            vg[i + (1 << b)] = vg[i] + L.Eg[b];
            vh[i + (1 << b)] = vh[i] + L.Eh[b];
        }
    }
}

// Expand one parent with a group of LP lanes.  The sink is called once per valid successor:
//   sink(mask, idx, posn, gnew, hnew)   idx = rank of mask among the valid masks (ascending)
template <int N, class Sink>
__device__ __forceinline__ void pg_expand_parent(const DevProblem &p, const PairMeta *meta, int *s_grp, const int (&pos)[N],
                                                 int g, int parenti, int sub, unsigned gmask, Sink &sink)
{
    using C = ExpCfg<N>;
    const int *s_hhg = s_grp + 8 * C::P;
    const int *s_hhh = s_hhg + C::H;
    ExpLane<N> L;
    pg_expand_prepare<N>(p, meta, s_grp, pos, g, parenti, sub, gmask, L);

    int posn[N];
#pragma unroll
    for (int i = 0; i < C::A; i++) posn[i] = pos[i] + ((sub >> i) & 1);
    const int full = (1 << N) - 1;
    const bool interior = L.alive == full;

    for (int u = 0; u < (1 << C::UB); u++) {
        int vg[1 << C::IB], vh[1 << C::IB];
        pg_expand_block<N>(L, u, vg, vh);
#pragma unroll
        for (int b = 0; b < C::UB; b++) posn[C::A + C::IB + b] = pos[C::A + C::IB + b] + ((u >> b) & 1);
#pragma unroll
        for (int i = 0; i < (1 << C::IB); i++) {
            const int high = (u << C::IB) | i;
            const int mask = (high << C::A) | sub;
#pragma unroll
            for (int b = 0; b < C::IB; b++) posn[C::A + b] = pos[C::A + b] + ((i >> b) & 1);
            if (mask == 0) continue;
            if (!interior && (mask & ~L.alive)) continue;
            const int idx = interior ? mask - 1 : pg_mask_rank<N>(mask, L.alive);
            sink(mask, idx, posn, vg[i] + s_hhg[high], vh[i] + s_hhh[high]);
        }
    }
    __syncwarp(gmask);
}
