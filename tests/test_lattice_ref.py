"""The exhaustive lattice reference and the table checker of tests/lattice_ref.py, on the CPU:
  * the level-order DP over the whole lattice reproduces the reference's optima;
  * the serial A*'s settled set (oracle po_astar_settled) is exactly {v : g*(v) + h(v) < F}, with g == g* and optimal
    moves, after a small budget and at the goal;
  * check_table finds nothing wrong with the table an exact A* leaves, and reports each kind of planted fault."""
import functools

import numpy as np
import pytest

from conftest import FIXTURES, KNOWN_OPT
from lattice_ref import Lattice, check_table, closed_walks, dense_lookup, lattice_g, rescore_chains
from oracle import oracle as O

NAMES = ["PF08184", "test", "test2"]


@functools.lru_cache(maxsize=None)
def reference(name):
    seqs = FIXTURES[name]
    P = O.Problem(seqs)
    lat = Lattice(seqs, P.int_weights())
    g, par = lattice_g(lat)
    return P, lat, g, par


@pytest.mark.parametrize("name", NAMES)
def test_lattice_dp_reproduces_known_optimum(name):
    P, lat, g, _ = reference(name)
    assert g[-1] == KNOWN_OPT[name]
    assert lat.h(np.zeros((1, lat.n)))[0] <= g[-1] <= lat.upper_bound()


@pytest.mark.parametrize("budget", [40, 0])
@pytest.mark.parametrize("name", NAMES)
def test_oracle_settled_set_is_exact(name, budget):
    P, lat, g, _ = reference(name)
    F, pos, gs, par = P.astar_settled(budget)
    res = P.astar(budget, want_rows=False)
    assert len(pos) <= res["closed_size"]
    if budget == 0:
        assert res["finished"] == 1 and F >= g[-1] and len(pos) > 0
    h_all = lat.h(lat.unflat(np.arange(lat.size)))
    want = np.flatnonzero(g + h_all < F)
    got = lat.flat(pos)
    assert np.array_equal(np.sort(got), want)
    assert np.array_equal(gs, g[got])
    nz = pos.any(axis=1)
    pb = (par[nz, None] >> np.arange(lat.n)) & 1
    u = pos[nz].astype(np.int64) - pb
    assert (u >= 0).all()
    assert np.array_equal(g[lat.flat(u)] + lat.edge_cost(u, par[nz]), gs[nz])


def exact_astar_table(lat, g, par, F):
    """The table an exact A* with a consistent heuristic holds once its least open f is F: closed with g* and an optimal
    move below F, every successor of those open with its best relaxation."""
    h = lat.h(lat.unflat(np.arange(lat.size)))
    state = np.zeros(lat.size, dtype=np.int64)
    gt = np.full(lat.size, -1, dtype=np.int64)
    pt = np.full(lat.size, -1, dtype=np.int64)
    closed = np.flatnonzero(g + h < F)
    state[closed], gt[closed], pt[closed] = 2, g[closed], par[closed]
    cpos = lat.unflat(closed)
    terms = lat.pair_terms(cpos)
    for m in lat.masks:
        ok = np.all(cpos + lat.bits[m - 1] <= lat.lens, axis=1)
        w = closed[ok] + lat.mstride[m - 1]
        cand = g[closed[ok]] + lat.mask_cost([t[ok] for t in terms], int(m))
        upd = (state[w] != 2) & ((state[w] == 0) | (cand < gt[w]))  # w is unique within one move
        w, cand = w[upd], cand[upd]
        state[w], gt[w], pt[w] = 1, cand, m
    return state, gt, pt


def open_f(lat, state, gt):
    o = np.flatnonzero(state == 1)
    return int((gt[o] + lat.h(lat.unflat(o))).min())


def planted(lat, g, par, F):
    state, gt, pt = exact_astar_table(lat, g, par, F)
    return state.copy(), gt.copy(), pt.copy()


@pytest.mark.parametrize("name", ["PF08184", "test"])
def test_checker_accepts_exact_table_and_reports_planted_faults(name):
    P, lat, g, par = reference(name)
    fs = np.unique(g + lat.h(lat.unflat(np.arange(lat.size))))
    F0 = int(fs[np.count_nonzero(fs <= g[-1]) // 2 + 1])  # half-way through the f layers up to the optimum
    state, gt, pt = exact_astar_table(lat, g, par, F0)
    F = open_f(lat, state, gt)
    assert F >= F0
    allpos = lat.unflat(np.arange(lat.size))
    gstar = lambda p: g[lat.flat(p)]
    ub = 1 << 62  # this table keeps every successor of a closed node

    def run(st, gg, pp, F_=F):
        return check_table(dense_lookup(lat, st, gg, pp), lat, allpos, F_, ub, gstar=gstar)

    assert run(state, gt, pt) == []
    h = lat.h(allpos)
    closed = np.flatnonzero((state == 2) & allpos.any(axis=1))
    opn = np.flatnonzero(state == 1)
    rng = np.random.default_rng(7)
    v = int(closed[np.argmax(allpos[closed].sum(axis=1))])  # a deep settled node

    faults = {}
    s, a, b = planted(lat, g, par, F0); a[v] += 1; faults["settled g + 1"] = (s, a, b)
    s, a, b = planted(lat, g, par, F0); s[v] = 0; a[v] = b[v] = -1; faults["settled node dropped"] = (s, a, b)
    s, a, b = planted(lat, g, par, F0); s[v] = 1; faults["settled node marked open"] = (s, a, b)
    # a move into v that is not optimal
    pv = allpos[v]
    bad_moves = [int(m) for m in lat.masks if np.all(pv >= lat.bits[m - 1])
                 and g[v - lat.mstride[m - 1]] + lat.edge_cost(pv - lat.bits[m - 1], m)[0] != g[v]]
    assert bad_moves
    s, a, b = planted(lat, g, par, F0); b[v] = bad_moves[0]; faults["parenti not optimal"] = (s, a, b)
    o = int(rng.choice(opn))
    s, a, b = planted(lat, g, par, F0); a[o] = g[o] - 1; faults["open g below g*"] = (s, a, b)
    # an open successor of a closed node whose relaxation makes it required, dropped
    w = int(rng.choice(opn))
    s, a, b = planted(lat, g, par, F0); s[w] = 0; a[w] = b[w] = -1; faults["successor dropped"] = (s, a, b)
    for what, (s, a, b) in faults.items():
        assert run(s, a, b), what


def test_walks_and_chains_on_exact_table():
    P, lat, g, par = reference("test")
    F0 = int(np.median(g + lat.h(lat.unflat(np.arange(lat.size)))))
    state, gt, pt = exact_astar_table(lat, g, par, F0)
    F = open_f(lat, state, gt)
    look = dense_lookup(lat, state, gt, pt)
    nodes, depth = closed_walks(look, lat, F, 16, 3)
    assert depth.min() > 0 and len(nodes) > 16
    assert np.array_equal(rescore_chains(look, lat, nodes), g[lat.flat(nodes)])
    assert check_table(look, lat, nodes, F, 1 << 62) == []
    gt2 = gt.copy()
    far = lat.flat(nodes[np.argmax(nodes.sum(axis=1))])[0]
    gt2[far] += 1
    look2 = dense_lookup(lat, state, gt2, pt)
    assert check_table(look2, lat, nodes, F, 1 << 62)
