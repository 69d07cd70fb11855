"""Layered search (pg_search_layered): exact costs and alignments, the top-level passes number for number against the NumPy
reference (tests/layered_ref.py), both reconstruction knobs, incumbents, budgets, refusals and the CLI."""
import json
import subprocess

import numpy as np
import pytest

from conftest import CASES, KNOWN_OPT, WIDE_CASES, weighted_sp_score
from lattice_ref import Lattice, lattice_g
from layered_ref import Layered
from test_gpu_weighted import BIN, c_star
from test_layered_ref import LATTICES

ALL = dict(CASES)
ALL.update(WIDE_CASES)
CAP = 1 << 24
SMALL_LAT = ["test", "PF08184", "rag7s", "rag6", "one4", "one5"]
_refs = {}


def lattice_ref(name):
    if name not in _refs:
        from oracle import oracle as O
        seqs = LATTICES[name]
        lat = Lattice(seqs, O.Problem(seqs).int_weights())
        _refs[name] = (lat, int(lattice_g(lat)[0][-1]))
    return _refs[name]


def optimum(name):
    return KNOWN_OPT[name] if name in KNOWN_OPT else c_star(name)


def check_rows(seqs, G, r):
    assert r["finished"] == 1, r
    assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"] == r["f"] == r["lower_bound"]
    assert r["align_len"] == len(r["rows"][0])


@pytest.fixture(autouse=True)
def release_memory():
    yield
    try:
        import mpi_pastar_msa_b200 as m
        m.release_cached_memory()
    except Exception:
        pass


# ---- 1. the optimum, and an alignment that re-scores to it
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ALL))
def test_layered_cost_and_alignment(gpu_lib, name):
    seqs = ALL[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.layered_search(table_capacity=CAP)
    check_rows(seqs, G, r)
    assert r["g"] == optimum(name)
    st = r["layered"]
    assert st["iterations"] >= 1 and st["first_bound"] <= st["last_bound"] and st["passes"] > st["iterations"] - 1
    assert r["rounds"] == st["levels"] and st["peak_bytes"] > 0


# ---- 2. the top-level passes equal the reference's, and repeat
@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL_LAT)
def test_layered_counters_match_reference(gpu_lib, name):
    lat, cstar = lattice_ref(name)
    ref = Layered(lat).run(want_moves=False)
    with gpu_lib.PastarGPU(LATTICES[name]) as G:
        G.build_pair_tables()
        a = G.layered_search(table_capacity=1 << 16, want_rows=False)
        b = G.layered_search(table_capacity=1 << 16, want_rows=False)
        c = G.layered_search(table_capacity=1 << 16)
    assert a["g"] == ref.cstar == cstar and a["align_len"] == 0 and "rows" not in a
    st = a["layered"]
    top = ref.top
    assert (st["iterations"], st["first_bound"], st["last_bound"]) == (len(top), top[0]["U"], top[-1]["U"])
    assert st["top_expansions"] == top[-1]["expansions"]
    for k in ("expansions", "generated", "inserted"):
        assert a[k] == sum(p[k] for p in top), k
    assert a["rounds"] == sum(p["levels"] for p in top)
    assert st["max_level_nodes"] == max(p["max_level_nodes"] for p in top)
    assert st["max_held"] == max(p["max_held"] for p in top)
    for k in ("expansions", "generated", "inserted", "rounds", "g"):
        assert a[k] == b[k], k
    assert a["layered"] == b["layered"]
    check_rows(LATTICES[name], G, c)
    for k in ("iterations", "first_bound", "last_bound", "top_expansions"):
        assert c["layered"][k] == st[k], k


# ---- 3. the reconstruction knobs
@pytest.mark.gpu
@pytest.mark.parametrize("knob", ["PG_LAYERED_DEEP", "PG_LAYERED_RETAIN"])
@pytest.mark.parametrize("name", SMALL_LAT)
def test_layered_knobs(gpu_lib, name, knob, monkeypatch):
    lat, cstar = lattice_ref(name)
    monkeypatch.setenv(knob, "1")
    with gpu_lib.PastarGPU(LATTICES[name]) as G:
        G.build_pair_tables()
        r = G.layered_search(table_capacity=1 << 16)
    check_rows(LATTICES[name], G, r)
    assert r["g"] == cstar
    if knob == "PG_LAYERED_RETAIN":
        assert r["layered"]["depth"] == 1 and r["layered"]["passes"] == r["layered"]["iterations"] + 1
    else:  # down to single moves: one relay pass per move at most, plus the top level's
        assert r["layered"]["passes"] - r["layered"]["iterations"] + 1 >= r["align_len"]


# ---- 4. incumbents and the budget
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["PF08184", "fam5x60", "fam7x30", "kinase"])
def test_layered_incumbents(gpu_lib, name):
    seqs = ALL[name]
    cstar = optimum(name)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        h0 = int(G.calculate_h(np.zeros((1, len(seqs)), dtype=np.uint16))[0])
        w2 = G.search(table_capacity=1 << 22, batch_target=16384, weight=2)["rows"]
        G.search_set_weight(1, 1)
        opt = G.layered_search(table_capacity=CAP)
        r = G.layered_search(table_capacity=CAP, incumbent=opt["rows"])
        assert r["finished"] == 2 and r["g"] == r["lower_bound"] == cstar and r["rows"] == opt["rows"]
        u = G.score_alignment(w2)
        r = G.layered_search(table_capacity=CAP, incumbent=w2)
        assert r["g"] == r["lower_bound"] == cstar and r["finished"] == (2 if u == cstar else 1)
        assert r["layered"]["last_bound"] <= u
        if r["finished"] == 1:
            check_rows(seqs, G, r)
        G.search_set_incumbent(None)
        for budget in (1, opt["expansions"] // 3, opt["expansions"] - 1):
            r = G.layered_search(table_capacity=CAP, max_expansions=max(1, budget))
            assert r["finished"] == 0 and "rows" not in r, budget
            assert h0 <= r["lower_bound"] <= cstar, (budget, r["lower_bound"])


# ---- 5. refusals, each with its status code and nothing clamped
@pytest.mark.gpu
def test_layered_refusals(gpu_lib):
    seqs = CASES["PF08184"]
    with gpu_lib.PastarGPU(seqs) as G:
        with pytest.raises(gpu_lib.PastarError) as e:
            G.layered_search()
        assert e.value.code == 5  # no pair tables
        G.build_pair_tables()
        G.search_set_weight(2048, 1024)
        with pytest.raises(gpu_lib.PastarError) as e:
            G.layered_search()
        assert e.value.code == 1
        G.search_set_weight(1, 1)
        G.search_begin()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.layered_search()
        assert e.value.code == 5
        G.search_end()
    with gpu_lib.PastarGPU(CASES["kinase"]) as G:  # levels of thousands of coordinates
        G.build_pair_tables()
        for cap in (6, 600):  # one and a hundred coordinates per level
            with pytest.raises(gpu_lib.PastarError) as e:
                G.layered_search(table_capacity=cap)
            assert e.value.code == 4, cap
    with gpu_lib.PastarGPU(seqs, gap_open=40) as G:
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.layered_search()
        assert e.value.code == 3
    wide = ["ACDEFGHIKLMNPQRSTVWY" * 10] * 16  # 16 x 8 key bits = 128: the context takes it, the search does not
    with gpu_lib.PastarGPU(wide, weights=None) as G:
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.layered_search()
        assert e.value.code == 3


# ---- 6. memory: the level tables against the A* table.  Measured on one B200 (profiles/r05_layered.json): at most 37 554
# coordinates held at once against A*'s 6 862 687 inserted (1 / 183); the limit leaves room for a different bound schedule.
@pytest.mark.gpu
def test_layered_holds_a_fraction_of_astar(gpu_lib):
    seqs = CASES["kinase"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        a = G.search(table_capacity=1 << 27, batch_target=16384, want_rows=False)
        r = G.layered_search(table_capacity=CAP, want_rows=False)
    assert a["g"] == r["g"] == KNOWN_OPT["kinase"]
    assert r["layered"]["max_held"] * 100 <= a["inserted"], (r["layered"]["max_held"], a["inserted"])


# ---- 7. CLI
def _cli(args):
    return subprocess.run([BIN] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)


def _fasta(path, rows):
    path.write_text("".join(">s%d\n%s\n" % (i, s) for i, s in enumerate(rows)))
    return str(path)


def test_cli_layered_refusals(tmp_path):
    fa = _fasta(tmp_path / "x.fasta", ["ACDE", "ACDF", "ACEE"])
    for a in (["--anytime", "2,1"], ["--weight", "2"], ["-g", "2"]):
        r = _cli(["--layered"] + a + [fa])
        assert r.returncode == 1 and "cannot be combined" in r.stderr.decode(), (a, r.returncode, r.stderr.decode())
    assert "--layered" in _cli([]).stdout.decode()


@pytest.mark.gpu
def test_cli_layered_pf08184(gpu_lib, tmp_path):
    seqs = CASES["PF08184"]
    fa = _fasta(tmp_path / "pf.fasta", seqs)
    js = tmp_path / "m.json"
    r = _cli(["--layered", "--weight", "1", "--metrics_json", str(js), fa])
    assert r.returncode == 0, r.stderr.decode()
    out = r.stdout.decode()
    line = next(l for l in out.split("\n") if l.startswith("Final Score:"))
    assert int(line.split("g - ")[1].split()[0]) == 24450
    assert "Lower bound: 24450" in out and "\nLayered: " in out
    d = json.load(open(js))
    assert d["finished"] == 1 and d["g"] == d["lower_bound"] == 24450
    assert d["layered"]["iterations"] >= 1 and d["layered"]["passes"] >= d["layered"]["iterations"]
