"""The layered search's NumPy reference (tests/layered_ref.py) against the exhaustive lattice optimum, on the CPU: the cost
is optimal, the rebuilt alignment re-scores to it, and the deepest recursion and retain-everything agree."""
import functools
import random

import numpy as np
import pytest

from conftest import AA, FIXTURES, weighted_sp_score
from lattice_ref import Lattice, lattice_g
from layered_ref import Layered, rows_of
from oracle import oracle as O


def ragged(lens, seed):
    r = random.Random(seed)
    return ["".join(r.choice(AA) for _ in range(L)) for L in lens]


# the reference fixtures that fit the exhaustive DP in seconds, ragged lattices as test_gpu_bench_state.py's, and inputs
# with length-1 sequences (levels of one node, moves that leave a sequence finished at once)
LATTICES = {k: FIXTURES[k] for k in ("test", "PF08184")}
LATTICES.update({"rag4": ragged((30, 32, 34, 31), 41), "rag6": ragged((9, 10, 11, 9, 10, 8), 61),
                 "rag7": ragged((6, 7, 5, 8, 6, 7, 5), 71), "rag7s": ragged((3, 4, 2, 5, 3, 4, 2), 72),
                 "one3": ["W", "C", "K"], "one4": ["A", "MKV", "W", "QR"], "one5": ragged((1, 12, 1, 9, 14), 5)})


@functools.lru_cache(maxsize=None)
def reference(name):
    seqs = LATTICES[name]
    w = O.Problem(seqs).int_weights()
    lat = Lattice(seqs, w)
    g, _ = lattice_g(lat)
    return seqs, w, lat, int(g[-1])


def check(name, **kw):
    seqs, w, lat, cstar = reference(name)
    L = Layered(lat, **kw).run()
    assert L.finished == 1 and L.cstar == cstar == L.lb
    rows = rows_of(seqs, L.moves)
    assert weighted_sp_score(seqs, w, rows) == cstar
    us = [p["U"] for p in L.top]
    assert us == sorted(set(us)) and us[0] == min(int(lat.h(np.zeros((1, lat.n)))[0]) + 1, L.cap)
    assert all(p["fmin"] is not None and p["fmin"] < q for p, q in zip(L.top, us[1:]))
    return L


@pytest.mark.parametrize("name", sorted(LATTICES))
def test_layered_cost_is_the_lattice_optimum(name):
    L = check(name)
    assert L.passes >= len(L.top)


@pytest.mark.parametrize("name", ["test", "rag7s", "rag6", "one4", "one5"])
def test_deepest_recursion_and_retain_all_agree(name):
    deep, whole = check(name, deep=True), check(name, retain_all=True)
    assert deep.cstar == whole.cstar
    assert [p["U"] for p in deep.top] == [p["U"] for p in whole.top]
    assert deep.depth >= whole.depth == 1
    # deep: every move is the crossing move of a relay pass (the last top-level pass's, or a reconstruction pass's)
    assert deep.passes - len(deep.top) + 1 >= len(deep.moves)


@pytest.mark.parametrize("name", ["PF08184", "rag7s"])
def test_incumbent_bounds(name):
    seqs, w, lat, cstar = reference(name)
    opt = Layered(lat, incumbent_cost=cstar).run()          # nothing is cheaper than the optimum
    assert opt.finished == 2 and opt.lb == cstar
    worse = Layered(lat, incumbent_cost=cstar + 500).run()  # a worse incumbent still finds C*
    assert worse.finished == 1 and worse.cstar == cstar
    assert all(p["U"] <= cstar + 500 for p in worse.top)
