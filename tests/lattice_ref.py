"""Exhaustive references for the search table and the checker that compares a table with them.

Under the reference cost model (GapOpen = GapExtension = GapGap = 30, Cost.h:13; PAM250 as cost; the pairwise reverse-DP
heuristic) h is consistent.  So for an exact search, with F the least f of any live open entry after the rounds run:
  1. soundness: every node in the table has g >= g*; every node but the origin has its predecessor v - parenti in the
     table, with g(v) >= g(u) + c(u, parenti);
  2. settledness: every node with g* + h < F is closed with g == g*, and its parenti is an optimal move;
  3. relaxation: every in-lattice successor w = v + m of a closed v with g(v) + c(v, m) + h(w) below the search's bound
     is in the table with g(w) <= g(v) + c(v, m);
  4. Bellman: for a settled v every predecessor u found in the table has g(u) + c(u, v) >= g(v).
check_table tests these through any `lookup` (pos -> state 0/1/2, g, parenti), against the exhaustive lattice optimum
(lattice_g) or against a serial A*'s settled set, and returns every violation it finds.

The edge cost is c(u, m) = sum over x < y of w_int[x][y] * t_xy, t_xy = cost90[seq_x[u_x], seq_y[u_y]] when x and y
both move and 30 otherwise (Node.cpp:129-152): the residues read are those at the predecessor's coordinate."""
import numpy as np

GAP = 30


class Lattice:
    """Cost model of one input: pair terms, heuristic tables, mask strides."""

    def __init__(self, seqs, w_int):
        from oracle import oracle as O
        self.seqs = [s if isinstance(s, str) else s.decode() for s in seqs]
        self.n = n = len(self.seqs)
        self.w = np.asarray(w_int, dtype=np.int64).reshape(n, n)
        self.lens = np.array([len(s) for s in self.seqs], dtype=np.int64)
        self.shape = tuple(int(l) + 1 for l in self.lens)
        self.size = int(np.prod(self.shape))
        self.strides = np.array([int(np.prod(self.shape[i + 1:])) for i in range(n)], dtype=np.int64)
        self.cost90 = O.cost_table().astype(np.int64)
        self.pairs = [(x, y) for x in range(n - 1) for y in range(x + 1, n)]
        # codes[x][i] = residue i of sequence x; index len holds the NUL the reference reads there (never a moving residue)
        self.codes = [np.array([ord(c) for c in s] + [0], dtype=np.int64) for s in self.seqs]
        P = O.Problem(self.seqs, self.w.astype(np.int32))
        self.tables = [P.table(k).astype(np.int64) for k in range(len(self.pairs))]
        P.close()
        self.masks = np.arange(1, 1 << n)
        self.bits = (self.masks[:, None] >> np.arange(n)) & 1                      # (2^n - 1, n)
        self.mstride = self.bits @ self.strides                                       # flat offset of each move
        both = [[k for k, (x, y) in enumerate(self.pairs) if (m >> x) & 1 and (m >> y) & 1] for m in self.masks]
        self.mask_pairs = both
        wsum = sum(int(self.w[x, y]) for x, y in self.pairs)
        self.mask_const = np.array([GAP * (wsum - sum(int(self.w[self.pairs[k]]) for k in b)) for b in both], dtype=np.int64)
        self._H = None
        if self.size <= 1 << 24:  # small lattices: h of every node once, then one gather per query
            self._H = self.h(self.unflat(np.arange(self.size)))

    def h(self, pos):
        pos = np.asarray(pos, dtype=np.int64).reshape(-1, self.n)
        if self._H is not None:
            return self._H[self.flat(pos)]
        out = np.zeros(len(pos), dtype=np.int64)
        for k, (x, y) in enumerate(self.pairs):
            out += self.tables[k][pos[:, x], pos[:, y]] * self.w[x, y]
        return out

    def pair_terms(self, u):
        """w_xy * cost90 of the residues at u, per pair: the match terms of a move out of u."""
        u = np.asarray(u, dtype=np.int64).reshape(-1, self.n)
        r = [self.codes[x][np.minimum(u[:, x], self.lens[x])] for x in range(self.n)]
        return [self.cost90[r[x], r[y]] * self.w[x, y] for x, y in self.pairs]

    def mask_cost(self, terms, m):
        """c(u, m) from pair_terms(u) for one move mask m (1 .. 2^n - 1)."""
        c = np.full(len(terms[0]) if terms else 1, self.mask_const[m - 1], dtype=np.int64)
        for k in self.mask_pairs[m - 1]:
            c = c + terms[k]
        return c

    def edge_cost(self, u, masks):
        """c(u, m) for every row of u and its mask (scalar or one per row), int64."""
        u = np.asarray(u, dtype=np.int64).reshape(-1, self.n)
        masks = np.broadcast_to(np.asarray(masks, dtype=np.int64), (len(u),))
        terms = self.pair_terms(u)
        out = np.zeros(len(u), dtype=np.int64)
        for m in np.unique(masks):
            sel = masks == m
            out[sel] = self.mask_cost([t[sel] for t in terms], int(m))
        return out

    def flat(self, pos):
        pos = np.asarray(pos, dtype=np.int64).reshape(-1, self.n)
        out = pos[:, 0] * self.strides[0]
        for i in range(1, self.n):
            out += pos[:, i] * self.strides[i]
        return out

    def unflat(self, idx):
        idx = np.asarray(idx, dtype=np.int64)
        return np.stack([(idx // self.strides[i]) % self.shape[i] for i in range(self.n)], axis=1)

    def upper_bound(self):
        """Cost of the all-advance alignment (column t moves every sequence with t < len): the search's UB."""
        total, pos = 0, np.zeros(self.n, dtype=np.int64)
        for t in range(int(self.lens.max())):
            m = int(sum(1 << i for i in range(self.n) if t < self.lens[i]))
            total += int(self.edge_cost(pos, m)[0])
            pos = pos + self.bits[m - 1]
        return total


def edge_cost(seqs, w_int, u, masks):
    return Lattice(seqs, w_int).edge_cost(u, masks)


def lattice_g(lat):
    """Exhaustive DP over the whole lattice in level order (level = sum of coordinates): (g*, one optimal parenti) per
    flat index.  The origin's parenti is the all-ones mask, as the search seeds it."""
    coords = lat.unflat(np.arange(lat.size))
    level = coords.sum(axis=1)
    order = np.argsort(level, kind="stable")
    bounds = np.searchsorted(level[order], np.arange(level.max() + 2))
    big = np.iinfo(np.int64).max // 4
    g = np.full(lat.size, big, dtype=np.int64)
    par = np.zeros(lat.size, dtype=np.int32)
    g[0], par[0] = 0, (1 << lat.n) - 1
    for L in range(1, int(level.max()) + 1):
        idx = order[bounds[L]:bounds[L + 1]]
        c = coords[idx]
        terms = lat.pair_terms(c - 1)  # the move's residues are those at the predecessor, c - 1 in every moving dim
        can = c >= 1
        best = np.full(len(idx), big, dtype=np.int64)
        arg = np.zeros(len(idx), dtype=np.int32)
        for m in lat.masks:
            ok = np.all(can[:, lat.bits[m - 1] == 1], axis=1)
            if not ok.any():
                continue
            cand = np.where(ok, g[np.where(ok, idx - lat.mstride[m - 1], 0)] + lat.mask_cost(terms, int(m)), big)
            better = cand < best
            best = np.where(better, cand, best)
            arg = np.where(better, m, arg)
        g[idx], par[idx] = best, arg
    return g, par


def dense_lookup(lat, state, g, par):
    """A lookup function over dense per-flat-index arrays (a whole lattice looked up once)."""
    def lookup(pos):
        f = lat.flat(pos)
        return state[f], g[f], par[f]
    return lookup


def _spread(sel, ii, flags):
    sel[:] = False
    sel[ii[flags]] = True
    return sel


def check_table(lookup, lat, pos, F, bound, gstar=None, F_set=None, limit=20):
    """Check invariants 1-4 (module docstring) on the nodes `pos` of a table read through `lookup`.

    F: the table's least live open f; bound: successors with g(v) + c + h(w) < bound must be present (UB + 1 in a run
    with no goal yet; g*(goal) in a finished one).  gstar: pos -> g* (int64, -1 where unknown), the reference the table is
    held to: the exhaustive lattice, or a serial A*'s settled set (then known exactly for g* + h < F_set).  Settledness is
    required for every known node with g* + h < F_set (default F); any table node with g + h < F_set must be known.
    Without gstar a node is taken as settled when it is closed with g + h < F.  Returns a list of violation strings
    (at most `limit` per kind, with a count of the rest)."""
    F_set = F if F_set is None else F_set
    pos = np.asarray(pos, dtype=np.int64).reshape(-1, lat.n)
    out, counts = [], {}

    def bad(kind, sel, fmt):
        k = int(np.count_nonzero(sel))
        if not k:
            return
        counts[kind] = counts.get(kind, 0) + k
        for i in np.flatnonzero(sel)[: max(0, limit - (counts[kind] - k))]:
            out.append("%s at %s: %s" % (kind, pos[i].tolist(), fmt(i)))

    st, g, par = (np.asarray(a, dtype=np.int64) for a in lookup(pos))
    h = lat.h(pos)
    present = st > 0
    origin = ~pos.any(axis=1)
    gs = np.asarray(gstar(pos), dtype=np.int64) if gstar else None

    # 1. soundness
    if gs is not None:
        bad("g below g*", present & (gs >= 0) & (g < gs), lambda i: "g %d < g* %d" % (g[i], gs[i]))
        bad("node below F_set missing from the reference", present & (gs < 0) & (g + h < F_set),
            lambda i: "g %d + h %d < %d" % (g[i], h[i], F_set))
    bad("origin g", present & origin & (g != 0), lambda i: "g %d" % g[i])
    nz = present & ~origin
    pm = np.where(nz, par, 0)
    pbits = (pm[:, None] >> np.arange(lat.n)) & 1
    okmove = nz & (pm > 0) & (pm < (1 << lat.n)) & np.all(pos >= pbits, axis=1)
    bad("parenti not a move into the node", nz & ~okmove, lambda i: "parenti %d" % par[i])
    u = pos - pbits
    ust, ug, _ = (np.asarray(a, dtype=np.int64) for a in lookup(np.where(okmove[:, None], u, 0)))
    cu = lat.edge_cost(np.where(okmove[:, None], u, 0), np.where(okmove, pm, 1))
    bad("predecessor missing", okmove & (ust == 0), lambda i: "v - parenti %s absent" % u[i].tolist())
    bad("g below predecessor + edge", okmove & (ust > 0) & (g < ug + cu),
        lambda i: "g %d < g(u) %d + c %d" % (g[i], ug[i], cu[i]))

    # 2. settledness
    if gs is not None:
        want = (gs >= 0) & (gs + h < F_set)
        bad("settled node absent", want & ~present, lambda i: "g* %d + h %d < F %d" % (gs[i], h[i], F_set))
        bad("settled node open", want & (st == 1), lambda i: "g %d, g* %d" % (g[i], gs[i]))
        bad("settled node with g != g*", want & (st == 2) & (g != gs), lambda i: "g %d, g* %d" % (g[i], gs[i]))
        gu = np.asarray(gstar(np.where(okmove[:, None], u, 0)), dtype=np.int64)
        opt = want & (st == 2) & okmove & ~origin
        bad("settled node's parenti not optimal", opt & ((gu < 0) | (gu + cu != gs)),
            lambda i: "g*(v - %d) %d + c %d != g* %d" % (par[i], gu[i], cu[i], gs[i]))
        settled = want & (st == 2)
    else:
        settled = (st == 2) & (g + h < F)
        bad("settled node's parenti not tight", settled & okmove & (ust > 0) & (ug + cu != g),
            lambda i: "g(u) %d + c %d != g %d" % (ug[i], cu[i], g[i]))

    # 3. relaxation (closed nodes) and 4. Bellman (settled nodes), one move mask at a time over the nodes it applies to
    closed = st == 2
    fterms = lat.pair_terms(pos)
    bterms = lat.pair_terms(np.maximum(pos - 1, 0))
    room = ((pos < lat.lens) << np.arange(lat.n)).sum(axis=1)    # the dims a move out of the node may advance
    back = ((pos >= 1) << np.arange(lat.n)).sum(axis=1)          # the dims a move into the node may come from
    for m in lat.masks:
        ii = np.flatnonzero(closed & ((room & m) == m))
        if len(ii):
            w = pos[ii] + lat.bits[m - 1]
            cand = g[ii] + lat.mask_cost([t[ii] for t in fterms], int(m))
            hw = lat.h(w)
            keep = cand + hw < bound
            ii, w, cand, hw = ii[keep], w[keep], cand[keep], hw[keep]
        if len(ii):
            wst, wg, _ = (np.asarray(a, dtype=np.int64) for a in lookup(w))
            sel = np.zeros(len(pos), dtype=bool)
            bad("successor of a closed node missing", _spread(sel, ii, wst == 0),
                lambda i, m=m: "move %d, g %d" % (m, g[i] + lat.edge_cost(pos[i], m)[0]))
            bad("successor g above the closed node's relaxation", _spread(sel, ii, (wst > 0) & (wg > cand)),
                lambda i, m=m: "move %d: g(w) %d > g %d + c %d" % (m, lookup(pos[i] + lat.bits[m - 1])[1][0], g[i],
                                                                  lat.edge_cost(pos[i], m)[0]))
            if gs is not None:  # a successor cheap enough to be settled must be known to the reference
                wgs = np.asarray(gstar(w), dtype=np.int64)
                bad("successor below F_set missing from the reference", _spread(sel, ii, (wst > 0) & (wgs < 0) & (wg + hw < F_set)),
                    lambda i, m=m: "move %d" % m)
        ii = np.flatnonzero(settled & ((back & m) == m))
        if len(ii):
            ust2, ug2, _ = (np.asarray(a, dtype=np.int64) for a in lookup(pos[ii] - lat.bits[m - 1]))
            cb = lat.mask_cost([t[ii] for t in bterms], int(m))
            bad("Bellman: a predecessor beats the settled g", _spread(np.zeros(len(pos), dtype=bool), ii, (ust2 > 0) & (ug2 + cb < g[ii])),
                lambda i, m=m: "move %d from g(u) %d" % (m, lookup(pos[i] - lat.bits[m - 1])[1][0]))
    for kind, k in counts.items():
        if k > limit:
            out.append("%s: %d in all" % (kind, k))
    return out


def rescore_chains(lookup, lat, pos):
    """Follow parenti from every node of `pos` back to the origin in lockstep and sum the edge costs: the g each node's
    stored path re-scores to (-1 where the chain breaks: an absent node or a move out of the lattice)."""
    cur = np.asarray(pos, dtype=np.int64).reshape(-1, lat.n).copy()
    total = np.zeros(len(cur), dtype=np.int64)
    alive = cur.any(axis=1)
    for _ in range(int(lat.lens.sum()) + 1):
        if not alive.any():
            break
        st, _, par = (np.asarray(a, dtype=np.int64) for a in lookup(cur[alive]))
        idx = np.flatnonzero(alive)
        pbits = (np.maximum(par, 0)[:, None] >> np.arange(lat.n)) & 1
        ok = (st > 0) & (par > 0) & np.all(cur[idx] >= pbits, axis=1)
        broken = idx[~ok]
        total[broken], alive[broken] = -1, False
        idx, pbits, par = idx[ok], pbits[ok], par[ok]
        u = cur[idx] - pbits
        total[idx] += lat.edge_cost(u, par)
        cur[idx] = u
        alive[idx] = cur[idx].any(axis=1)
    total[alive] = -1
    return total


def closed_walks(lookup, lat, F, k, seed, max_steps=None):
    """k random walks in lockstep from the origin through settled nodes (closed, g + h < F): each step looks up all
    2^N - 1 successors of every walk in one call and moves to a random settled one; a walk stops when there is none.
    Returns the visited nodes (unique, K x N) and each walk's depth."""
    rng = np.random.default_rng(seed)
    cur = np.zeros((k, lat.n), dtype=np.int64)
    depth = np.zeros(k, dtype=np.int64)
    alive = np.ones(k, dtype=bool)
    seen = [cur.copy()]
    steps = int(lat.lens.sum()) if max_steps is None else max_steps
    for _ in range(steps):
        idx = np.flatnonzero(alive)
        if not len(idx):
            break
        w = cur[idx][:, None, :] + lat.bits[None, :, :]                 # (k, 2^N - 1, N)
        inl = np.all(w <= lat.lens, axis=2)
        wq = np.where(inl[:, :, None], w, 0).reshape(-1, lat.n)
        st, g, _ = (np.asarray(a, dtype=np.int64) for a in lookup(wq))
        ok = (inl.reshape(-1) & (st == 2) & (g + lat.h(wq) < F)).reshape(len(idx), -1)
        has = ok.any(axis=1)
        alive[idx[~has]] = False
        idx, ok, w = idx[has], ok[has], w[has]
        if not len(idx):
            break
        pick = np.array([rng.choice(np.flatnonzero(r)) for r in ok])
        cur[idx] = w[np.arange(len(idx)), pick]
        depth[idx] += 1
        seen.append(cur[idx].copy())
    return np.unique(np.concatenate(seen), axis=0), depth
