"""The beam search's NumPy reference (tests/beam_ref.py) against the exhaustive lattice optimum, on the CPU: the lower bound
is at most the optimum and the optimum at most the alignment's cost, the traced alignment re-scores to it, a beam as wide
as the widest level is exact, the cut keeps exactly the W least (f, packed key), and the phase loop's incumbent rules."""
import functools

import numpy as np
import pytest

from beam_ref import Beam, beam_pass, cut, key_bits
from conftest import weighted_sp_score
from layered_ref import rows_of
from test_layered_ref import LATTICES, reference


@functools.lru_cache(maxsize=None)
def widest(name):
    lat = reference(name)[2]
    return int(np.bincount(lat.unflat(np.arange(lat.size)).sum(axis=1)).max())


@pytest.mark.parametrize("W", [1, 2, 3, 7, 64, "widest"])
@pytest.mark.parametrize("name", sorted(LATTICES))
def test_beam_bounds_the_lattice_optimum(name, W):
    seqs, w, lat, cstar = reference(name)
    W = widest(name) if W == "widest" else W
    o = beam_pass(lat, W, lat.upper_bound() + 1)
    assert o["lb"] <= cstar
    assert o["kept"] == o["expansions"] and o["max_candidates"] >= 1
    if o["reached"]:
        assert cstar <= o["goal_g"]
        assert weighted_sp_score(seqs, w, rows_of(seqs, o["moves"])) == o["goal_g"]
    if W >= widest(name):
        assert o["dropped"] == 0 and o["drop_fmin"] is None
        assert o["reached"] and o["goal_g"] == o["lb"] == cstar


def test_cut_resolves_a_tie_class_that_straddles_the_width():
    rng = np.random.default_rng(7)
    kb, n = 6, 4
    pos = np.unique(rng.integers(0, 1 << kb, size=(400, n)), axis=0)
    f = rng.integers(100, 104, size=len(pos))           # four f classes of about 100 entries each
    packed = [sum(int(p[i]) << (i * kb) for i in range(n)) for p in pos]
    ranked = sorted(range(len(pos)), key=lambda j: (int(f[j]), packed[j]))
    for W in (1, 37, int((f == 100).sum()) + 5, len(pos) - 1):
        assert int((f <= f[ranked[W - 1]]).sum()) > W or W == len(pos) - 1  # the class at the cut straddles W
        keep, drop = cut(f, pos, W)
        assert sorted(keep.tolist()) == sorted(ranked[:W]) and len(drop) == len(pos) - W


def test_cut_on_a_lattice_level_matches_the_packed_key():
    seqs, w, lat, cstar = reference("rag6")
    kb = key_bits(lat)
    idx = np.flatnonzero(lat.unflat(np.arange(lat.size)).sum(axis=1) == 20)
    pos = lat.unflat(idx)
    f = lat.h(pos) // 1000                              # coarse f: wide tie classes
    packed = [sum(int(p[i]) << (i * kb) for i in range(lat.n)) for p in pos]
    ranked = sorted(range(len(pos)), key=lambda j: (int(f[j]), packed[j]))
    for W in (1, 50, len(pos) // 2):
        assert sorted(cut(f, pos, W)[0].tolist()) == sorted(ranked[:W])


@pytest.mark.parametrize("name", ["PF08184", "rag7s", "one4"])
def test_beam_incumbent_and_phase_loop(name):
    seqs, w, lat, cstar = reference(name)
    full = widest(name)
    opt = Beam(lat, [full], incumbent_cost=cstar).run()    # nothing is cheaper than the optimum: the incumbent stands
    assert opt.finished == 2 and opt.lb == cstar == opt.g and opt.best_phase == -1
    B = Beam(lat, [1, 2, full, full]).run()                # proved by the full width at the latest: the last never runs
    assert B.finished == 1 and B.g == B.lb == cstar and len(B.phases) <= 3
    before = B.phases[:-1]                                  # the loop stops at the first phase that proves the optimum
    assert not any(p["reached"] and p["goal_g"] <= max(q["lb"] for q in before) for p in before)
    assert weighted_sp_score(seqs, w, rows_of(seqs, B.moves)) == cstar
    gs = [p["goal_g"] for p in B.phases if p["reached"]]
    assert gs == sorted(set(gs), reverse=True)              # each phase that reaches the goal strictly improves
    assert all(p["U"] == (B.phases[0]["U"] if k == 0 else min([q["goal_g"] for q in B.phases[:k] if q["reached"]] or [p["U"]]))
               for k, p in enumerate(B.phases))
    worse = Beam(lat, [1], incumbent_cost=cstar + 10 ** 6).run()
    assert worse.finished in (1, 2) and worse.lb <= cstar <= worse.g
