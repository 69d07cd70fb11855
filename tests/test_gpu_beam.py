"""Beam search (pg_search_beam): every phase number for number against the NumPy reference (tests/beam_ref.py), alignments
that re-score to their cost with a certified bound on every reference case, the width schedule, incumbents, refusals and
the CLI.  About a minute on one B200."""
import json
import subprocess

import numpy as np
import pytest

from beam_ref import Beam
from conftest import CASES, KNOWN_OPT, WIDE_CASES, weighted_sp_score
from test_gpu_layered import ALL, SMALL_LAT, _cli, _fasta, lattice_ref, optimum
from test_gpu_weighted import BIN
from test_layered_ref import LATTICES

CAP = 1 << 24


@pytest.fixture(autouse=True)
def release_memory():
    yield
    try:
        import mpi_pastar_msa_b200 as m
        m.release_cached_memory()
    except Exception:
        pass


def check_alignment(seqs, G, r, cstar):
    assert r["finished"] in (1, 2), r
    assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"] == r["f"]
    assert r["align_len"] == len(r["rows"][0])
    assert r["lower_bound"] <= cstar <= r["g"], (r["lower_bound"], cstar, r["g"])
    assert r["finished"] == 2 or r["g"] == r["lower_bound"] == cstar


# ---- 1. every phase equals the reference's, number for number, and repeats
@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL_LAT)
def test_beam_phases_match_reference(gpu_lib, name):
    lat, cstar = lattice_ref(name)
    seqs = LATTICES[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        for W in (1, 2, 5, 64, 4096):
            ref = Beam(lat, [W]).run()
            o = ref.phases[0]
            a = G.beam_search([W], table_capacity=1 << 18)
            G.search_set_incumbent(None)  # an improved alignment stays the context's incumbent
            b = G.beam_search([W], table_capacity=1 << 18, want_rows=False)
            G.search_set_incumbent(None)
            assert len(a["phases"]) == 1
            p = a["phases"][0]
            assert (p["g"] >= 0) == o["reached"], W
            assert p["g"] == o["goal_g"] and p["lower_bound"] == o["lb"] == a["lower_bound"], W
            for k in ("expansions", "generated", "inserted", "levels", "kept", "dropped"):
                assert p[k] == o[k], (W, k, p[k], o[k])
            st = a["beam"]
            assert (st["phases"], st["kept"], st["dropped"], st["levels"]) == (1, o["kept"], o["dropped"], o["levels"])
            assert st["max_candidates"] == o["max_candidates"], W
            assert a["finished"] == ref.finished and a["g"] == ref.g, W
            if ref.finished:
                check_alignment(seqs, G, a, cstar)
            for k in ("finished", "g", "lower_bound", "expansions", "generated", "inserted", "rounds"):
                assert a[k] == b[k], (W, k)
            assert a["phases"] == b["phases"] and a["beam"] == b["beam"]


# ---- 2. the reference cases at a large width: an alignment that re-scores to g, and LB <= C* <= g
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ALL))
def test_beam_alignment_and_bound(gpu_lib, name):
    seqs = ALL[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.beam_search([4096], table_capacity=CAP)
    check_alignment(seqs, G, r, optimum(name))
    st = r["beam"]
    assert st["best_phase"] == 0 and st["peak_bytes"] > 0 and st["retained"] >= st["kept"]
    assert r["rounds"] == st["levels"] == sum(len(s) for s in seqs)


# ---- 3. the width schedule: the early stop on proof, per-phase results, a budget that runs out inside a phase
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rag7s", "rag6"])
def test_beam_schedule(gpu_lib, name):
    lat, cstar = lattice_ref(name)
    ref = Beam(lat, [1, 3, 1 << 20, 1 << 20]).run()
    with gpu_lib.PastarGPU(LATTICES[name]) as G:
        G.build_pair_tables()
        r = G.beam_search([1, 3, 1 << 20, 1 << 20], table_capacity=1 << 18)
        assert r["finished"] == 1 and r["g"] == r["lower_bound"] == cstar
        assert [(p["width"], p["g"], p["lower_bound"]) for p in r["phases"]] == \
            [(p["width"], p["goal_g"], p["lb"]) for p in ref.phases]
        assert r["beam"]["phases"] == len(ref.phases) <= 3 and r["beam"]["best_phase"] == ref.best_phase
        G.search_set_incumbent(None)
        full = G.beam_search([1 << 20], table_capacity=1 << 18, want_rows=False)
        G.search_set_incumbent(None)
        for budget in (1, full["expansions"] // 2):
            b = G.beam_search([1 << 20], table_capacity=1 << 18, max_expansions=budget)
            assert b["finished"] == 0 and "rows" not in b and b["phases"] == [], budget
            assert b["lower_bound"] <= cstar and b["expansions"] >= budget
    assert full["finished"] == 1 and full["g"] == cstar


# ---- 4. incumbents: a strict improvement, or the incumbent returned
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["PF08184", "fam7x30", "kinase"])
def test_beam_incumbents(gpu_lib, name):
    seqs = ALL[name]
    cstar = optimum(name)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        opt = G.search(table_capacity=1 << 24, batch_target=16384)
        w3 = G.search(table_capacity=1 << 22, batch_target=16384, weight=3)
        G.search_set_weight(1, 1)
        r = G.beam_search([1 << 16], incumbent=opt["rows"], table_capacity=CAP)
        assert r["finished"] == 2 and r["g"] == cstar and r["rows"] == opt["rows"] and r["lower_bound"] <= cstar
        assert r["beam"]["best_phase"] == -1
        u = G.score_alignment(w3["rows"])
        r = G.beam_search([16, 4096], incumbent=w3["rows"], table_capacity=CAP)
        assert cstar <= r["g"] <= u and r["lower_bound"] <= cstar
        assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"]
        if r["g"] < u:  # a phase improved it: that phase's g, and it is the context's incumbent now
            assert r["beam"]["best_phase"] >= 0 and r["g"] == r["phases"][r["beam"]["best_phase"]]["g"] < u
            assert all(p["g"] < u for p in r["phases"] if p["g"] >= 0)
        else:
            assert r["finished"] == 2 and r["rows"] == w3["rows"]
        G.search_set_incumbent(None)


# ---- 5. refusals, each with its status code
@pytest.mark.gpu
def test_beam_refusals(gpu_lib):
    seqs = CASES["PF08184"]
    with gpu_lib.PastarGPU(seqs) as G:
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([4])
        assert e.value.code == 5  # no pair tables
        G.build_pair_tables()
        for widths in ([], [0], [4, -1], [1] * 65):
            with pytest.raises(gpu_lib.PastarError) as e:
                G.beam_search(widths)
            assert e.value.code == 1, widths
        G.search_set_weight(2048, 1024)
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([4])
        assert e.value.code == 1
        G.search_set_weight(1, 1)
        G.search_begin()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([4])
        assert e.value.code == 5
        G.search_end()
    with gpu_lib.PastarGPU(CASES["fam7x30"]) as G:  # 31^7 = 2.75e10 coordinates: a beam as wide as the lattice
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([1 << 40])
        assert e.value.code == 4 and "2^32" in str(e.value)
        with pytest.raises(gpu_lib.PastarError) as e:  # 3.5 G retained nodes and 2^30-coordinate levels: > 180 GB
            G.beam_search([1 << 24])
        assert e.value.code == 4 and "free on the device" in str(e.value)
    with gpu_lib.PastarGPU(CASES["kinase"]) as G:
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([4096], table_capacity=600)  # a hundred candidates per level
        assert e.value.code == 4
    with gpu_lib.PastarGPU(seqs, gap_open=40) as G:
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([4])
        assert e.value.code == 3
    wide = ["ACDEFGHIKLMNPQRSTVWY" * 10] * 16  # 16 x 8 key bits = 128
    with gpu_lib.PastarGPU(wide, weights=None) as G:
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.beam_search([4])
        assert e.value.code == 3


# ---- 6. CLI
def test_cli_beam_refusals(tmp_path):
    fa = _fasta(tmp_path / "x.fasta", ["ACDE", "ACDF", "ACEE"])
    for a in (["--anytime", "2,1"], ["--weight", "2"], ["-g", "2"]):
        r = _cli(["--beam", "4"] + a + [fa])
        assert r.returncode == 1 and "cannot be combined" in r.stderr.decode(), (a, r.returncode, r.stderr.decode())
    for bad in ("0", "4,x", "-3", "4,,5", ",".join(["2"] * 65)):
        r = _cli(["--beam", bad, fa])
        assert r.returncode == 1 and "--beam" in r.stderr.decode(), (bad, r.stderr.decode())
    assert "--beam" in _cli([]).stdout.decode()


def _score(out):
    line = next(l for l in out.split("\n") if l.startswith("Final Score:"))
    return int(line.split("g - ")[1].split()[0])


@pytest.mark.gpu
def test_cli_beam_kinase(gpu_lib, tmp_path):
    seqs = CASES["kinase"]
    cstar = KNOWN_OPT["kinase"]
    fa = _fasta(tmp_path / "k.fasta", seqs)
    js = tmp_path / "m.json"
    r = _cli(["--beam", "4096,65536", "--metrics_json", str(js), fa])
    assert r.returncode == 0, r.stderr.decode()
    out = r.stdout.decode()
    assert "\nBeam: " in out
    d = json.load(open(js))
    g, lb = _score(out), d["lower_bound"]
    assert d["finished"] in (1, 2) and d["g"] == g == d["beam"]["g"] and lb <= cstar <= g
    assert [p["width"] for p in d["beam"]["phases"]] == [4096, 65536][:len(d["beam"]["phases"])]
    # the printed alignment re-scores to the printed score
    blocks = [l for l in out.split("\n") if l and set(l) <= set("ACDEFGHIKLMNPQRSTVWY-")]
    rows = ["".join(blocks[i::5]) for i in range(5)]
    with gpu_lib.PastarGPU(seqs) as G:
        assert G.score_alignment(rows) == g
    # --beam then --layered: the beam's alignment bounds the layered search, which still returns the optimum
    inc = _fasta(tmp_path / "inc.fasta", rows)
    r = _cli(["--beam", "4096", "--layered", "--metrics_json", str(js), fa])
    assert r.returncode == 0, r.stderr.decode()
    d = json.load(open(js))
    assert d["finished"] in (1, 2) and d["g"] == d["lower_bound"] == cstar
    assert d["layered"]["last_bound"] <= d["beam"]["g"] and "beam" in d and "\nLayered: " in r.stdout.decode()
    # --beam with --incumbent: never worse than the incumbent
    r = _cli(["--beam", "64", "--incumbent", inc, "--metrics_json", str(js), fa])
    assert r.returncode == 0, r.stderr.decode()
    d = json.load(open(js))
    assert d["incumbent"] == g and d["g"] <= g and d["lower_bound"] <= cstar
