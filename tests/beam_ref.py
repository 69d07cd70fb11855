"""NumPy restatement of the beam search (pg_search_beam, DESIGN.md §4.4d) on a lattice_ref.Lattice.

A phase of width W and bound U sweeps the lattice level by level (level = sum of the coordinates) from the origin.  A
successor x of an expanded node is kept when g + h < U; each level's entries are merged by the least (g, low), where low is
the parent's index in the retained array.  Before level d is expanded its entries are cut: when there are more than W, the W
least by (f = g + h, packed key) stay, the packed key being sum pos_i << (i kb) with kb the context's key_bits, compared as
an unsigned integer.  The others are dropped: counted, and the least f among them kept.  Every kept node is appended to the
retained array as (coordinate, g, parent index); the origin's parent is the sentinel 2^32 - 1.  The goal's parent index
leads back to the origin.

The phase's lower bound is min(g(goal) if it was reached, the least f dropped, U).  Phases run one per width, each with
U = the best alignment so far (the incumbent's cost, or the all-advance cost + 1), and stop once the largest lower bound
reaches the best cost.  finished: 1 when a phase found the alignment returned and the bound equals its cost, 2 for an
alignment with a gap or the incumbent unimproved, 0 when no alignment is known.

For a fixed width and bound the kept sets, their g, every counter, the goal's g and the bound do not depend on the order
of anything; the parent indices do, so among parents of equal g the GPU may trace another alignment of the same cost."""
import numpy as np

from layered_ref import _merge

SENTINEL = (1 << 32) - 1


def key_bits(lat):
    """The context's bits per coordinate in the packed key: the least kb with 2^kb > the longest sequence."""
    return max(1, int(lat.lens.max()).bit_length())


def cut(f, pos, W):
    """Indices of the W least entries by (f, packed key).  The packed key orders as the coordinates read from the last
    sequence to the first, each field being narrower than kb bits."""
    if len(f) <= W:
        return np.arange(len(f)), np.zeros(0, dtype=np.int64)
    order = np.lexsort(tuple(pos[:, i] for i in range(pos.shape[1])) + (f,))
    return order[:W], order[W:]


def beam_pass(lat, W, U):
    """One phase; returns a dict with reached, goal_g, moves (origin first) when reached, drop_fmin, lb and the counters."""
    n = lat.n
    D = int(lat.lens.sum())
    H = lat._H if lat._H is not None else lat.h(lat.unflat(np.arange(lat.size)))
    out = dict(reached=False, goal_g=-1, moves=None, drop_fmin=None, expansions=0, generated=0, inserted=1, levels=0,
               kept=0, dropped=0, max_candidates=0)
    pending = {0: [(lat.flat(np.zeros(n, dtype=np.int64)), np.array([SENTINEL], dtype=np.int64))]}
    ret_idx, ret_par = [], []
    for d in range(D):
        idx, val = _merge(pending.pop(d, []))
        if d:
            out["inserted"] += len(idx)
        out["max_candidates"] = max(out["max_candidates"], len(idx))
        g = val >> 32
        if len(idx):
            keep, drop = cut(g + H[idx], lat.unflat(idx), W)
            if len(drop):
                fd = int((g + H[idx])[drop].min())
                out["drop_fmin"] = fd if out["drop_fmin"] is None else min(out["drop_fmin"], fd)
                out["dropped"] += len(drop)
            idx, val, g = idx[keep], val[keep], g[keep]
        rid = np.arange(len(ret_idx), len(ret_idx) + len(idx), dtype=np.int64)
        ret_idx.extend(idx.tolist())
        ret_par.extend((val & 0xffffffff).tolist())
        k = len(idx)
        out["expansions"] += k
        out["kept"] += k
        out["levels"] += 1
        if k:
            pos = lat.unflat(idx)
            terms = lat.pair_terms(pos)
            for mi, m in enumerate(lat.masks):
                ok = np.all(pos + lat.bits[mi] <= lat.lens, axis=1)
                out["generated"] += int(ok.sum())
                if not ok.any():
                    continue
                ii = np.flatnonzero(ok)
                gn = g[ii] + lat.mask_cost([tt[ii] for tt in terms], int(m))
                child = idx[ii] + lat.mstride[mi]
                keep = gn + H[child] < U
                if keep.any():
                    lv2 = d + int(lat.bits[mi].sum())
                    pending.setdefault(lv2, []).append((child[keep], (gn[keep] << 32) | rid[ii][keep]))
        if not [l for l in pending if d < l <= d + n]:
            break
    else:  # level D holds the goal alone
        idx, val = _merge(pending.pop(D, []))
        out["inserted"] += len(idx)
        if len(idx) == 1:
            out["reached"], out["goal_g"] = True, int(val[0]) >> 32
            moves, cur, p = [], lat.lens.copy(), int(val[0]) & 0xffffffff
            while p != SENTINEL:
                q = lat.unflat(np.array([ret_idx[p]]))[0]
                step = cur - q
                assert np.all((step == 0) | (step == 1)) and step.any()
                moves.append(int((step << np.arange(n)).sum()))
                cur, p = q, ret_par[p]
            assert not cur.any()
            out["moves"] = moves[::-1]
    for l in list(pending):  # entries of levels never taken were still inserted
        out["inserted"] += len(_merge(pending.pop(l))[0])
    lb = U if out["drop_fmin"] is None else min(U, out["drop_fmin"])
    out["lb"] = min(lb, out["goal_g"]) if out["reached"] else lb
    return out


class Beam:
    """pg_search_beam on the CPU: run() gives the phases, the best alignment's moves, its cost, the bound and finished."""

    def __init__(self, lat, widths, incumbent_cost=None):
        self.lat, self.widths, self.incumbent_cost = lat, list(widths), incumbent_cost

    def run(self):
        lat = self.lat
        ub = lat.upper_bound()
        best, improved = self.incumbent_cost, False
        self.lb = int(lat.h(np.zeros((1, lat.n), dtype=np.int64))[0])
        self.phases, self.moves, self.best_phase = [], None, -1
        for k, W in enumerate(self.widths):
            if best is not None and self.lb >= best:
                break
            U = best if best is not None else ub + 1
            o = beam_pass(lat, W, U)
            o.update(width=W, U=U)
            self.phases.append(o)
            self.lb = max(self.lb, o["lb"])
            if o["reached"]:
                assert o["goal_g"] < U
                best, improved, self.moves, self.best_phase = o["goal_g"], True, o["moves"], k
        self.g = -1 if best is None else best
        self.finished = 0 if best is None else (1 if improved and self.lb >= best else 2)
        return self
