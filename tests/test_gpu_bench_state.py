"""The search table at the benchmarked batch (2^20 pops a round) and table size (2^30 coordinates: 2^32 value slots, slot
ids at the top of their uint32 range) checked node by node, not only through the final cost:
  * small lattices run to the end, then every node looked up and held to the exhaustive lattice optimum (lattice_ref);
  * bench.py's S7 state after its exact schedule, held to the serial A*'s settled set and walked deep into the settled
    region; S8 (two-word keys, 8-byte values) the same way;
  * finished solves at the benchmarked sizes, and the batched lookup against the single one.
The invariants are listed in tests/lattice_ref.py."""
import os
import random
import re
import time

import numpy as np
import pytest

from conftest import AA, FIXTURES, KNOWN_OPT, ROOT, WIDE_CASES, random_seqs, weighted_sp_score
from lattice_ref import Lattice, check_table, closed_walks, dense_lookup, lattice_g, rescore_chains
from oracle import oracle as O

BATCH, CAP = 1 << 20, 1 << 30  # bench.py's defaults


def ragged(lens, seed):
    r = random.Random(seed)
    return ["".join(r.choice(AA) for _ in range(L)) for L in lens]


# made-up ragged inputs of about a million lattice nodes; N = 7 is the benchmark's kernel instantiation
LATTICES = dict(FIXTURES)
LATTICES.update({"rag4": ragged((30, 32, 34, 31), 41), "rag6": ragged((9, 10, 11, 9, 10, 8), 61),
                 "rag7": ragged((6, 7, 5, 8, 6, 7, 5), 71), "rag7s": ragged((3, 4, 2, 5, 3, 4, 2), 72)})
_refs = {}


def lattice_ref(name):
    if name not in _refs:
        seqs = LATTICES[name]
        lat = Lattice(seqs, O.Problem(seqs).int_weights())
        _refs[name] = (lat,) + lattice_g(lat)
    return _refs[name]


@pytest.fixture(autouse=True)
def release_memory():
    """The benchmarked table holds about 40 GiB while a search runs; give it back after each test (shared device)."""
    yield
    try:
        import mpi_pastar_msa_b200 as m
        m.release_cached_memory()
    except Exception:
        pass


def gpu_lookup(G):
    return lambda pos: G.search_lookup_many(np.asarray(pos, dtype=np.int64).astype(np.uint16))


def test_bench_defaults_are_the_checked_sizes():
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert re.search(r'"--batch", type=int, default=1 << 20\b', src)
    assert re.search(r'"--table-capacity", type=int, default=1 << 30\b', src)


def run_to_end(G, batch, cap):
    G.search_begin(1, 0, cap, batch)
    for _ in range(100000):
        F, best, c = G.search_status()
        if F >= best:
            return F, best, c
        G.search_rounds(8)
    raise AssertionError("search did not finish")


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("name,batch,cap,valw", [
    ("PF08184", BATCH, CAP, "auto"), ("test2", BATCH, CAP, "auto"), ("test", BATCH, CAP, "auto"),
    ("rag4", BATCH, CAP, "auto"), ("rag6", BATCH, CAP, "auto"), ("rag7", BATCH, CAP, "auto"),
    ("PF08184", 1, 1 << 22, "auto"), ("rag7s", 1, 1 << 22, "auto"),
    ("PF08184", BATCH, CAP, "8"), ("rag7", BATCH, CAP, "8")])
def test_exhaustive_lattice(gpu_lib, name, batch, cap, valw, monkeypatch):
    if valw == "8":
        monkeypatch.setenv("PG_VALW", "8")
    lat, g, _ = lattice_ref(name)
    with gpu_lib.PastarGPU(LATTICES[name]) as G:
        G.build_pair_tables()
        F, best, c = run_to_end(G, batch, cap)
        assert best == g[-1]
        allpos = lat.unflat(np.arange(lat.size))
        st, gt, pt = G.search_lookup_many(allpos.astype(np.uint16))
    assert c["inserted"] == np.count_nonzero(st)  # every coordinate the search stored, found where the lattice has it
    errs = check_table(dense_lookup(lat, st, gt, pt), lat, allpos, F, best, gstar=lambda p: g[lat.flat(p)],
                       F_set=min(F, best))
    print("%s batch %d: %d lattice nodes, %d in the table, %d closed" % (name, batch, lat.size, np.count_nonzero(st),
                                                                       np.count_nonzero(st == 2)))
    assert not errs, "\n".join(errs)


def oracle_gstar(lat, pos, g):
    """pos -> g from a serial A*'s settled set, -1 for nodes outside it."""
    keys = lat.flat(pos)
    order = np.argsort(keys)
    keys, gs = keys[order], np.asarray(g, dtype=np.int64)[order]

    def gstar(p):
        k = lat.flat(p)
        i = np.minimum(np.searchsorted(keys, k), len(keys) - 1)
        return np.where(keys[i] == k, gs[i], -1)
    return gstar


def check_against_oracle_and_walks(G, lat, F, oracle, walks=64):
    """(a) the oracle's settled set, (b) settled nodes deep in the region, found by random walks; returns counts."""
    F_cpu, opos, og, _ = oracle
    assert F_cpu <= F
    look = gpu_lookup(G)
    ub = lat.upper_bound()
    errs = check_table(look, lat, opos, F, ub + 1, gstar=oracle_gstar(lat, opos, og), F_set=F_cpu)
    assert not errs, "\n".join(errs)
    nodes, depth = closed_walks(look, lat, F, walks, 12345)
    errs = check_table(look, lat, nodes, F, ub + 1)
    assert not errs, "\n".join(errs)
    st, g, _ = look(nodes)
    assert (st == 2).all()
    assert np.array_equal(rescore_chains(look, lat, nodes), g)
    return len(opos), len(nodes), int(depth.min()), int(depth.max())


@pytest.mark.gpu
@pytest.mark.slow
def test_s7_bench_state(gpu_lib):
    """bench.py --gpus 1 with its defaults: ramp-up in groups of 8 rounds, 10 warm-up rounds, 100 timed rounds (graph
    replay) and 100 profiled rounds (plain launches); then the state is checked."""
    seqs = random_seqs(7, 500, 12345)
    t0 = time.time()
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        G.search_begin(1, 0, CAP, BATCH)
        ramp = 0
        while True:
            before = G.search_status()[2]["pops"]
            G.search_rounds(8)
            ramp += 8
            if G.search_status()[2]["pops"] - before >= 8 * BATCH or ramp > 4000:
                break
        G.search_rounds(10)
        G.search_rounds(100)
        G.search_profile(True)
        G.search_rounds(100)
        G.search_profile(False)
        F, best, c = G.search_status()
        assert best == 2**31 - 1 and c["finished"] == 0
        t1 = time.time()
        lat = Lattice(seqs, G.w_int)
        oracle = O.Problem(seqs, G.w_int).astar_settled(100000)
        n_or, n_walk, dmin, dmax = check_against_oracle_and_walks(G, lat, F, oracle)
    print("S7: %d expansions on the device (%.1f s); %d oracle-settled nodes, %d walk nodes at depth %d-%d (%.1f s)"
          % (c["expansions"], t1 - t0, n_or, n_walk, dmin, dmax, time.time() - t1))


@pytest.mark.gpu
@pytest.mark.slow
def test_s8_wide_key_state(gpu_lib):
    seqs = random_seqs(8, 1000, 12345)
    with gpu_lib.PastarGPU(seqs, weights=None) as G:
        G.build_pair_tables()
        G.search_begin(1, 0, 1 << 28, 1 << 18)
        while G.search_status()[2]["expansions"] < 5000000:
            G.search_rounds(8)
        F, best, c = G.search_status()
        assert best == 2**31 - 1
        lat = Lattice(seqs, G.w_int)
        oracle = O.Problem(seqs, G.w_int).astar_settled(50000)
        n_or, n_walk, dmin, dmax = check_against_oracle_and_walks(G, lat, F, oracle)
    print("S8: %d expansions; %d oracle-settled nodes, %d walk nodes at depth %d-%d" % (c["expansions"], n_or, n_walk, dmin, dmax))


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("name", ["kinase", "fam10x100"])
def test_finished_solve_at_bench_sizes(gpu_lib, name):
    seqs = FIXTURES.get(name) or WIDE_CASES[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.search(table_capacity=CAP, batch_target=BATCH)
        assert r["finished"] == 1 and r["g"] == KNOWN_OPT[name]
        assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"]
        if name != "kinase":
            return
        # every node the serial A* settles in 200 k pops, below the optimum, is closed with the serial g
        F_cpu, opos, og, _ = O.Problem(seqs, G.w_int).astar_settled(200000)
        lat = Lattice(seqs, G.w_int)
        keep = og + lat.h(opos) < r["g"]
        st, g, _ = G.search_lookup_many(opos[keep])
        assert (st == 2).all() and np.array_equal(g, og[keep])
        print("kinase: %d oracle-settled nodes below the optimum closed with the serial g" % keep.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["S7", "S8", "S7-valw8"])
def test_lookup_many_matches_single_lookup(gpu_lib, what, monkeypatch):
    if what == "S7-valw8":
        monkeypatch.setenv("PG_VALW", "8")
    seqs = random_seqs(8, 1000, 12345) if what == "S8" else random_seqs(7, 500, 12345)
    with gpu_lib.PastarGPU(seqs, weights=None if what == "S8" else "altschul") as G:
        G.build_pair_tables()
        G.search_begin(1, 0, 1 << 24, 4096)
        G.search_rounds(64)
        rng = np.random.default_rng(5)
        n = G.n
        bits = (np.arange(1, 1 << n)[:, None] >> np.arange(n)) & 1
        near = np.cumsum(bits[rng.integers(0, len(bits), (2000, 8))], axis=1)[np.arange(2000), rng.integers(0, 8, 2000)]
        far = rng.integers(0, 400, (1000, n))
        pos = np.concatenate([near, far]).astype(np.uint16)
        st, g, par = G.search_lookup_many(pos)
        assert np.count_nonzero(st) > 100 and np.count_nonzero(st == 0) > 100
        for k in range(len(pos)):
            one = G.search_lookup(pos[k])
            if one is None:
                assert st[k] == 0 and g[k] == -1 and par[k] == -1
            else:
                assert st[k] in (1, 2) and (g[k], par[k]) == one
        bad = pos[:3].copy()
        bad[1, 2] = G.lens[2] + 1
        with pytest.raises(gpu_lib.PastarError) as e:
            G.search_lookup_many(bad)
        assert e.value.code == 1
        G.search_end()
        with pytest.raises(gpu_lib.PastarError):
            G.search_lookup_many(pos[:3])
