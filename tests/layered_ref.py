"""NumPy restatement of the layered search (pg_search_layered, DESIGN.md §4.4c) on a lattice_ref.Lattice.

A pass sweeps the box [s, t] level by level (level = sum of the coordinates) from s with g(s) = g0.  A successor x of an
expanded node is kept when it lies in the box and g + h < U (strict) or g + h <= U; each level's entries are merged by
the least (g, low).  low is the move into x in retain mode; in relay mode it is the move when it crosses `mid`
(parent level <= mid < x's level) and the parent's low otherwise, and the nodes of levels mid + 1 .. mid + N entered by
a crossing move get a relay id.  In-box successors that fail only the bound feed f_min, f_max and a histogram.

The top level runs strict passes with U_0 = min(h(origin) + 1, cap), cap = the incumbent's cost or the all-advance cost
+ 1.  A pass that reaches the goal has found C* = g(goal).  Otherwise C* >= f_min, and the next bound is the least bin edge
U + (b + 1) w such that the pruned records of bins 0 .. b number at least floor(sqrt(expansions x generated)) of the
pass, else the top of the bins U + 2047 w, or f_min + 1 if that is higher; at most cap.  The bins have width w = max(1, ceil(2 (U - h0) / 2047)), the
last also holds everything above them.  f_min >= cap proves the incumbent optimal.

The alignment is rebuilt from the successful pass's relay x (entered from p = x - mask): solve(origin, p), the move,
solve(x, goal).  solve(s, t) runs a non-strict pass with U = C* over the box and recurses on its relay, or, when the box
spans at most R levels + 1, runs one retain pass and follows the stored moves back from t.  R = 4 (N + 1); deep: R = 1;
retain_all: R = D + 1 and one retain pass over the whole lattice.

The GPU's counters of the top-level passes (expansions, generated, inserted, levels, the bounds) equal these number for
number: for a fixed bound the set of expanded nodes and their g do not depend on thread order.  Relay ids do, so when
several relays tie the GPU may rebuild another optimal alignment than this reference."""
import numpy as np

NB = 2048
RELAY_BASE = 1 << 16


def _merge(parts):
    """(flat, value) pairs of one level -> unique flat indices with the least value each."""
    if not parts:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    idx = np.concatenate([p[0] for p in parts])
    val = np.concatenate([p[1] for p in parts])
    order = np.lexsort((val, idx))
    idx, val = idx[order], val[order]
    first = np.ones(len(idx), dtype=bool)
    first[1:] = idx[1:] != idx[:-1]
    return idx[first], val[first]


def level_pass(lat, s, t, g0, U, strict, mid, retain, W=1):
    """One pass; returns a dict with reached, goal_g, the relay (x, g, mask) when reached in relay mode, fmin, fmax, hist,
    hist_w, the counters, and (retain) the merged levels."""
    n = lat.n
    s, t = np.asarray(s, dtype=np.int64), np.asarray(t, dtype=np.int64)
    ls, lt = int(s.sum()), int(t.sum())
    H = lat._H if lat._H is not None else lat.h(lat.unflat(np.arange(lat.size)))
    out = dict(reached=False, goal_g=-1, fmin=None, fmax=None, hist=np.zeros(NB, dtype=np.int64), hist_w=W, expansions=0,
               generated=0, inserted=1, levels=0, max_level_nodes=0, max_held=0)
    low0 = (1 << n) - 1 if retain else RELAY_BASE
    pending = {ls: [(lat.flat(s), np.array([(g0 << 32) | low0], dtype=np.int64))]}
    merged = {}
    relay = []
    pop = np.array([bin(m).count("1") for m in lat.masks])
    fmin, fmax = None, None

    def take(d):
        idx, val = _merge(pending.pop(d, []))
        if d != ls:
            out["inserted"] += len(idx)
        if not retain and mid < d <= mid + n:
            cross = (val & 0xffffffff) < RELAY_BASE
            for k in np.flatnonzero(cross):
                relay.append((int(idx[k]), int(val[k])))
                val[k] = (val[k] & ~0xffffffff) | (RELAY_BASE + len(relay) - 1)
        merged[d] = (idx, val)
        return idx, val

    for d in range(ls, lt):
        idx, val = take(d)
        k = len(idx)
        out["expansions"] += k
        out["levels"] += 1
        out["max_level_nodes"] = max(out["max_level_nodes"], k)
        if k:
            pos = lat.unflat(idx)
            g = val >> 32
            low = val & 0xffffffff
            terms = lat.pair_terms(pos)
            for mi, m in enumerate(lat.masks):
                b = lat.bits[mi]
                ok = np.all(pos + b <= lat.lens, axis=1)
                out["generated"] += int(ok.sum())
                inbox = ok & np.all(pos + b <= t, axis=1)
                if not inbox.any():
                    continue
                ii = np.flatnonzero(inbox)
                gn = g[ii] + lat.mask_cost([tt[ii] for tt in terms], int(m))
                child = idx[ii] + lat.mstride[mi]
                f = gn + H[child]
                fail = f >= U if strict else f > U
                if fail.any():
                    ff = f[fail]
                    fmin = int(ff.min()) if fmin is None else min(fmin, int(ff.min()))
                    fmax = int(ff.max()) if fmax is None else max(fmax, int(ff.max()))
                    np.add.at(out["hist"], np.minimum((ff - U) // W, NB - 1), 1)
                keep = ~fail
                if not keep.any():
                    continue
                lv2 = d + int(pop[mi])
                if retain or (d <= mid < lv2):
                    lo = np.full(int(keep.sum()), m, dtype=np.int64)
                else:
                    lo = low[ii][keep]
                pending.setdefault(lv2, []).append((child[keep], (gn[keep] << 32) | lo))
        ahead = [l for l in pending if d < l <= d + n]
        if retain:
            held = out["inserted"] + sum(len(_merge(pending[l])[0]) for l in pending if l > ls)
        else:
            held = k + sum(len(_merge(pending[l])[0]) for l in ahead)
        out["max_held"] = max(out["max_held"], held)
        if not ahead:
            break
    else:  # not stopped early: level lt holds t alone
        take(lt)
    if lt in merged and len(merged[lt][0]) == 1:
        v = int(merged[lt][1][0])
        out["reached"], out["goal_g"] = True, v >> 32
        if not retain:
            x, rv = relay[(v & 0xffffffff) - RELAY_BASE]
            out["relay"] = (lat.unflat(np.array([x]))[0], rv >> 32, rv & 0xffffffff)
    # pending entries of levels never taken were still inserted
    for l in list(pending):
        out["inserted"] += len(_merge(pending.pop(l))[0])
    out["fmin"], out["fmax"] = fmin, fmax
    if retain:
        out["merged"] = merged
    return out


def bin_width(U, h0):
    return max(1, -(-2 * max(1, U - h0) // (NB - 1)))


def next_bound(o, U, cap):
    w = o["hist_w"]
    cum = np.cumsum(o["hist"][:-1])
    hit = np.flatnonzero(cum >= max(1, int(np.sqrt(float(o["expansions"]) * float(o["generated"])))))
    if len(hit):
        return min(cap, U + (int(hit[0]) + 1) * w)
    return min(cap, max(U + (NB - 1) * w, o["fmin"] + 1))


class Layered:
    """pg_search_layered on the CPU: run() gives C*, the alignment's moves, the top-level passes and the stats."""

    def __init__(self, lat, incumbent_cost=None, deep=False, retain_all=False):
        self.lat = lat
        n = lat.n
        self.D = int(lat.lens.sum())
        self.cap = incumbent_cost if incumbent_cost is not None else lat.upper_bound() + 1
        self.R = self.D + 1 if retain_all else (1 if deep else 4 * (n + 1))
        self.retain_all = retain_all
        self.passes, self.top, self.depth = 0, [], 0

    def _pass(self, *a, W=1):
        self.passes += 1
        return level_pass(self.lat, *a, W=W)

    def run(self, want_moves=True):
        lat = self.lat
        origin, goal = np.zeros(lat.n, dtype=np.int64), lat.lens.copy()
        h0 = int(lat.h(origin[None])[0])
        self.lb, self.cstar, self.finished = h0, None, 0
        if h0 >= self.cap:
            self.finished, self.lb = 2, self.cap
            return self
        U = min(h0 + 1, self.cap)
        while True:
            o = self._pass(origin, goal, 0, U, True, self.D // 2, False, W=bin_width(U, h0))
            self.top.append(dict(U=U, expansions=o["expansions"], generated=o["generated"], inserted=o["inserted"],
                                 levels=o["levels"], max_level_nodes=o["max_level_nodes"], max_held=o["max_held"],
                                 fmin=o["fmin"]))
            if o["reached"]:
                self.cstar, self.finished, self.lb = o["goal_g"], 1, o["goal_g"]
                break
            fmin = self.cap if o["fmin"] is None else o["fmin"]
            self.lb = max(self.lb, min(fmin, self.cap))
            if fmin >= self.cap:
                assert self.cap != lat.upper_bound() + 1, "no path below the all-advance cost"
                self.finished, self.lb = 2, self.cap
                return self
            nU = next_bound(o, U, self.cap)
            assert nU > fmin and nU > U
            U = nU
        self.moves = None
        if want_moves:
            if self.retain_all:
                self.moves = self.solve(origin, goal, 0, self.cstar, 1)
            else:
                self.moves = self.split(origin, goal, 0, self.cstar, o, 0)
        return self

    def solve(self, s, t, gs, gt, depth):
        ls, lt = int(s.sum()), int(t.sum())
        if ls == lt:
            return []
        self.depth = max(self.depth, depth)
        retain = lt - ls + 1 <= self.R
        o = self._pass(s, t, gs, self.cstar, False, (ls + lt) // 2, retain)
        assert o["reached"] and o["goal_g"] == gt, (s, t, o["goal_g"], gt)
        if not retain:
            return self.split(s, t, gs, gt, o, depth)
        moves, cur = [], t.copy()
        while int(cur.sum()) > ls:
            idx, val = o["merged"][int(cur.sum())]
            k = np.searchsorted(idx, self.lat.flat(cur)[0])
            m = int(val[k]) & 0xffffffff
            moves.append(m)
            cur = cur - self.lat.bits[m - 1]
        assert np.array_equal(cur, s)
        return moves[::-1]

    def split(self, s, t, gs, gt, o, depth):
        x, gx, m = o["relay"]
        p = x - self.lat.bits[m - 1]
        gp = gx - int(self.lat.edge_cost(p, m)[0])
        return self.solve(s, p, gs, gp, depth + 1) + [m] + self.solve(x, t, gx, gt, depth + 1)


def rows_of(seqs, moves):
    """The alignment spelled by move masks (origin first)."""
    at = [0] * len(seqs)
    rows = [[] for _ in seqs]
    for m in moves:
        for i, sq in enumerate(seqs):
            if (m >> i) & 1:
                rows[i].append(sq[at[i]])
                at[i] += 1
            else:
                rows[i].append("-")
    return ["".join(r) for r in rows]
