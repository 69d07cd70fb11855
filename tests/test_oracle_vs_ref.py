"""CPU: the C oracle against the reference itself (oracle/_ref/pastar_ref = unmodified reference sources compiled in
place).  Without that build the reference's values come from tests/golden/ref_comparisons.json.gz (tests/refdata.py)."""
import numpy as np
import pytest

from conftest import CASES, family_seqs, random_parents, random_seqs
from oracle import oracle as O
from oracle import refio as R
import refdata as D

RAND = {"r5x50": random_seqs(5, 50, 41), "f4x90": family_seqs(4, 90, 42, 0.2, 0.05), "f16x5": CASES["fam16x5"],
        "f14x6": CASES["fam14x6"], "r3x998": random_seqs(3, 998, 43)}


@pytest.mark.parametrize("name", list(RAND))
def test_dump(name):
    seqs = RAND[name]
    assert D.digest(O.cost_table()) == D.dump(seqs)["cost"]
    _check_dump(seqs)


def _check_dump(seqs):
    d = D.dump(seqs)
    assert O.weights(seqs).view(np.uint32).ravel().tolist() == d["weights"]
    k = 0
    for i in range(len(seqs) - 1):
        for j in range(i + 1, len(seqs)):
            t = O.pair_table(seqs[i], seqs[j])
            assert [list(t.shape), D.digest(t)] == [d["shapes"][k], d["tables"][k]], (i, j)
            k += 1


def _check_neigh(P, seqs, pos, g, par, vs, ht, sh):
    ref = D.neigh(seqs, pos, g, par, vs, ht, sh)
    for k in range(len(pos)):
        mine = P.get_neigh(pos[k], g[k], par[k], vs, ht, sh)
        assert int(g[k]) + P.calculate_h(pos[k]) == ref["fpar"][k]
        assert [len(mine), D.digest(mine)] == [ref["count"][k], ref["records"][k]], (k, vs, ht, sh)


@pytest.mark.parametrize("name", ["r5x50", "f4x90", "f14x6"])
def test_get_neigh(name):
    seqs = RAND[name]
    n = len(seqs)
    P = O.Problem(seqs)
    pos, g, par = random_parents(seqs, 6 if n <= 10 else 2, 5)
    for (vs, ht, sh) in [(1, "FZORDER", 12), (7, "FZORDER", 1), (4, "PZORDER", 3), (3, "FSUM", 2), (6, "PSUM", 0)]:
        _check_neigh(P, seqs, pos, g, par, vs, ht, sh)


def test_astar_and_partitioned_driver():
    seqs = RAND["f4x90"]
    P = O.Problem(seqs)
    a = P.astar(want_rows=False)
    r = D.astar(seqs)
    assert [a["g"], a["expansions"], a["generated"]] == r
    if D.live():  # the reference's own T-thread hash-partitioned driver (PAStar.cpp:319-547 restated): same optimal cost
        p = R.pastar(seqs, 4)
        assert p["finished"] == 1 and p["g"] == r[0]


def _edge_inputs():
    import random
    al = "ACDEFGHIKLMNPQRSTVWY"
    rng = random.Random(11)
    return {
        "len1_mixed": ["A", "C", "DE", "F", "GHI"],                     # sequences of one residue: 2-row tables
        "identical3": ["ACDEFG"] * 3,                                    # zero-cost diagonal, all ties
        "ragged6": ["".join(rng.choice(al) for _ in range(l)) for l in (1, 2, 17, 3, 40, 9)],
        "unset_pam_rows": ["ABXXJOU", "BJXBOXAA", "UOJACD", "ACDXB"],    # SURVEY F2: B, J, O, U, X cost 0 against everything
        "ragged9": ["".join(rng.choice(al) for _ in range(rng.randint(1, 12))) for _ in range(9)],
        "ragged10": ["".join(rng.choice(al) for _ in range(rng.randint(1, 8))) for _ in range(10)],
    }


@pytest.mark.parametrize("name", list(_edge_inputs()))
def test_edge_inputs(name):
    """Tables, weights, calculate_h, getNeigh records and owners on degenerate inputs, parents on the lattice borders
    (start, goal, goal - 1, alternating corners) included; serial A* counters where the search is small."""
    import random
    seqs = _edge_inputs()[name]
    n = len(seqs)
    _check_dump(seqs)
    P = O.Problem(seqs)
    rng = random.Random(3)
    fin = [len(s) for s in seqs]
    pos = [[0] * n, fin[:], [max(0, f - 1) for f in fin], [f if i % 2 else 0 for i, f in enumerate(fin)]]
    pos += [[rng.randint(0, f) for f in fin] for _ in range(4)]
    pos = np.array(pos, dtype=np.uint16)
    g = np.arange(len(pos), dtype=np.int32) * 37
    par = np.array([(1 << n) - 1, 1, 2, 3, 1, (1 << n) - 2, 5, 4], dtype=np.int32)
    for (vs, ht, sh) in [(1, "FZORDER", 12), (8, "FZORDER", 0), (4, "PZORDER", 1), (3, "FSUM", 2), (5, "PSUM", 0)]:
        _check_neigh(P, seqs, pos, g, par, vs, ht, sh)
    if n <= 5:
        a = P.astar(want_rows=False)
        assert [a["g"], a["expansions"], a["generated"]] == D.astar(seqs)


@pytest.mark.parametrize("seed", range(24))
def test_seeded_fuzz(seed):
    """Random small problems (N in 3..10, lengths 1..30, random or related sequences), random parents anywhere in the
    lattice incl. its faces, a random hash / shift / partition count: weights, tables, h and every getNeigh record."""
    import random
    rng = random.Random(1000 + seed)
    n = rng.choice([3, 4, 5, 6, 7, 8, 9, 10])
    if rng.random() < 0.5:
        seqs = ["".join(rng.choice("ACDEFGHIKLMNPQRSTVWY") for _ in range(rng.randint(1, 30))) for _ in range(n)]
    else:
        seqs = family_seqs(n, rng.randint(2, 30), 2000 + seed, sub=rng.choice([0.05, 0.3]), indel=rng.choice([0.0, 0.1]))
    _check_dump(seqs)
    P = O.Problem(seqs)
    fin = [len(s) for s in seqs]
    pos = np.array([[rng.choice([0, f, rng.randint(0, f)]) for f in fin] for _ in range(5)], dtype=np.uint16)
    g = np.array([rng.randint(0, 100000) for _ in range(5)], dtype=np.int32)
    par = np.array([rng.randint(1, (1 << n) - 1) for _ in range(5)], dtype=np.int32)
    vs, ht, sh = rng.choice([1, 2, 3, 4, 8, 16, 64]), rng.choice(["FZORDER", "PZORDER", "FSUM", "PSUM"]), rng.randint(0, 21)
    _check_neigh(P, seqs, pos, g, par, vs, ht, sh)
