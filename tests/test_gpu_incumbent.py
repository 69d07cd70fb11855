"""Incumbent-bounded and anytime search: with a known alignment of cost U every search keeps only what can beat U, and
either returns a cheaper alignment (finished 1) or reports that none exists (finished 2, the incumbent returned; an
exact search then has lower bound == U, a proof of optimality).  pg_search_anytime restarts weighted search with falling
weights, each phase bounded by the best alignment so far."""
import json
import subprocess

import pytest

from conftest import CASES, weighted_sp_score
from test_gpu_weighted import BIN, FAMILY, FAMILY_CAP, INT_MAX, REOPEN_STORM, SMALL, c_star

KINASE_OPT = 421546
ANYTIME = (2, 1.25, 1)  # the default schedule of PastarGPU.anytime_search


def exact_rows(G, batch=16384, cap=1 << 22):
    r = G.search(table_capacity=cap, batch_target=batch)
    assert r["finished"] == 1
    return r


def weighted_rows(m, seqs, w=2, cap=1 << 22):
    """The alignment of a w-weighted search at batch 16384 (no reopening storm there), on a context of its own."""
    with m.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.search(table_capacity=cap, batch_target=16384, weight=w)
        assert r["finished"] == 1
        return r["rows"]


# ---- 1. scoring
@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
def test_score_alignment(gpu_lib, name):
    seqs = CASES[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = exact_rows(G)
        assert G.score_alignment(r["rows"]) == weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"]
        rows = list(r["rows"])
        c = next(k for k, ch in enumerate(rows[0]) if ch != "-")
        bad = {
            "residue": [rows[0][:c] + ("A" if rows[0][c] != "A" else "C") + rows[0][c + 1:]] + rows[1:],
            "length": [rows[0] + "-"] + rows[1:],
            "all-gap column": [row + "-" for row in rows],
            "row count": rows[:-1],
        }
        for what, b in bad.items():
            with pytest.raises(gpu_lib.PastarError) as e:
                G.score_alignment(b)
            assert e.value.code == 1, what
            with pytest.raises(gpu_lib.PastarError) as e:
                G.search_set_incumbent(b)
            assert e.value.code == 1, what


# ---- 2. the optimum as incumbent: proved
# kinase runs at batch 16384 only: the proof expands the ~4.6 M nodes with f < C*, one per round at batch 1
@pytest.mark.gpu
@pytest.mark.parametrize("name,batch", [(n, b) for n in SMALL for b in (1, 16384)] + [("kinase", 16384)])
def test_optimal_incumbent_is_proved(gpu_lib, name, batch):
    seqs = CASES[name]
    cap = 1 << 27 if name == "kinase" else 1 << 22
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        opt = exact_rows(G, cap=cap)
        assert opt["g"] == c_star(name)
        r = G.search(table_capacity=cap, batch_target=batch, incumbent=opt["rows"])
        assert r["finished"] == 2, r
        assert r["g"] == r["lower_bound"] == c_star(name)
        assert r["rows"] == opt["rows"]
        assert r["align_len"] == len(opt["rows"][0])


# ---- 3. the w = 2 alignment as incumbent: the optimum, with fewer coordinates stored
# upper limits of inserted (bounded) / inserted (unbounded) at batch 1; the measured ratios are in the test's docstring
INSERTED_RATIO = {"fam5x60": 0.5, "fam7x30": 0.8}


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
def test_weighted_incumbent_tightens_exact_search(gpu_lib, name):
    """Exact search at batch 1 (deterministic counters) with the w = 2 alignment (batch 16384) as incumbent: the optimum,
    and never more coordinates than the unbounded search.  Measured on one B200 (profiles/r04_anytime_sweep.json),
    inserted bounded / unbounded: fam5x60 6 492 / 14 553 = 0.45 with U = 102 429 = 1.019 C*; fam7x30 33 842 / 44 290 = 0.76
    with U = 169 215 = 1.033 C*.
    The w = 2 alignment is 3 % above the optimum there, where pruning by f >= U saves a quarter of the table, not half."""
    seqs = CASES[name]
    inc = weighted_rows(gpu_lib, seqs)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        u = G.score_alignment(inc)
        a = G.search(table_capacity=1 << 22, batch_target=1)
        b = G.search(table_capacity=1 << 22, batch_target=1, incumbent=inc)
    assert b["g"] == b["lower_bound"] == c_star(name) <= u
    assert b["finished"] == (2 if u == c_star(name) else 1)
    assert weighted_sp_score(seqs, G.w_int, b["rows"]) == b["g"]
    assert b["inserted"] <= a["inserted"], (b["inserted"], a["inserted"])
    if name in INSERTED_RATIO:
        assert b["inserted"] <= INSERTED_RATIO[name] * a["inserted"], (b["inserted"], a["inserted"])


# ---- 4. weighted search with an incumbent
@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
@pytest.mark.parametrize("weight", [1.25, 2])
def test_weighted_search_with_incumbent(gpu_lib, name, weight):
    """Incumbents: the optimum (nothing cheaper: finished 2) and the w = 4 alignment (often beaten: finished 1)."""
    seqs = CASES[name]
    cstar = c_star(name)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        opt = exact_rows(G)["rows"]
        seen = set()
        for inc in (opt, weighted_rows(gpu_lib, seqs, 4)):
            u = G.score_alignment(inc)
            r = G.search(table_capacity=1 << 22, batch_target=16384, weight=weight, incumbent=inc)
            assert r["finished"] in (1, 2), r
            seen.add(r["finished"])
            assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"] <= u
            if r["finished"] == 2:
                assert r["g"] == u and r["rows"] == inc
            else:
                assert r["g"] < u
            assert r["lower_bound"] <= cstar <= r["g"], (r["lower_bound"], cstar, r["g"])
            assert r["g"] * r["weight_den"] <= r["weight_num"] * r["lower_bound"], r
        assert 2 in seen


# ---- 5. budgeted bounded runs
@pytest.mark.gpu
def test_budgeted_bounded_kinase(gpu_lib):
    seqs = CASES["kinase"]
    inc = weighted_rows(gpu_lib, seqs, 2, 1 << 27)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        u = G.score_alignment(inc)
        assert u > KINASE_OPT
        r = G.search(table_capacity=1 << 27, batch_target=16384, max_expansions=100000, incumbent=inc, want_rows=False)
        assert r["finished"] == 0
        assert r["lower_bound"] <= KINASE_OPT <= u


@pytest.mark.gpu
@pytest.mark.parametrize("weight", [1, 2])
def test_budgeted_bounded_stepwise_partitioned(gpu_lib, weight):
    """The loop-back step-wise driver of test_gpu_weighted.py over two partitions, stopped at a budget."""
    seqs = CASES["kinase"]
    inc = weighted_rows(gpu_lib, seqs, 2, 1 << 27)
    Gs = []
    for r in range(2):
        G = gpu_lib.PastarGPU(seqs)
        G.build_pair_tables()
        G.configure_hash("FZORDER", 0)
        G.search_set_weight(*gpu_lib.weight_fraction(weight))
        G.search_set_incumbent(inc)
        G.search_begin(2, r, 1 << 26, 4096)
        Gs.append(G)
    u = Gs[0].score_alignment(inc)
    with pytest.raises(gpu_lib.PastarError) as e:  # not while a step-wise search is active
        Gs[0].search_set_incumbent(None)
    assert e.value.code == 5
    best = INT_MAX
    while True:
        for G in Gs:
            G.search_round(best)
        boxes = [[G.search_outbox(d) if d != r else (0, 0) for d in range(2)] for r, G in enumerate(Gs)]
        for r in range(2):
            for d in range(2):
                ptr, n = boxes[r][d]
                if n:
                    Gs[d].search_insert_dev(ptr, n)
        st = [G.search_status() for G in Gs]
        best = min(s[1] for s in st)
        if sum(s[2]["expansions"] for s in st) >= 50000 or min(s[0] for s in st) >= best:
            break
    lb = min(G.search_lower_bound() for G in Gs)
    assert best == INT_MAX or best < u
    assert lb <= KINASE_OPT <= u, (lb, u)
    for G in Gs:
        G.search_end()
        G.close()


# ---- 6. pg_multi_search
@pytest.mark.gpu
@pytest.mark.parametrize("name,parts,batch,ht,sh", [("fam5x60", 2, 256, "FZORDER", 0), ("fam8x20", 4, 4096, "PZORDER", 1)])
def test_multi_search_with_incumbent(gpu_lib, name, parts, batch, ht, sh):
    seqs = CASES[name]
    cstar = c_star(name)
    inc = weighted_rows(gpu_lib, seqs, 4)
    Gs = []
    for _ in range(parts):
        G = gpu_lib.PastarGPU(seqs)
        G.build_pair_tables()
        G.configure_hash(ht, sh)
        Gs.append(G)
    u = Gs[0].score_alignment(inc)
    tot, _ = gpu_lib.multi_search(Gs, table_capacity=1 << 22, batch_target=batch, incumbent=inc)
    assert tot["g"] == tot["lower_bound"] == cstar
    assert tot["finished"] == (2 if u == cstar else 1)
    assert weighted_sp_score(seqs, Gs[0].w_int, tot["rows"]) == cstar
    opt = tot["rows"]
    tot, per = gpu_lib.multi_search(Gs, table_capacity=1 << 22, batch_target=batch, incumbent=opt)
    assert tot["finished"] == 2 and all(p["finished"] == 2 for p in per)
    assert tot["g"] == tot["lower_bound"] == cstar and tot["rows"] == opt
    assert all(G.search_lower_bound() == cstar for G in Gs)
    Gs[1].search_set_incumbent(inc if u != cstar else None)
    with pytest.raises(gpu_lib.PastarError) as e:
        gpu_lib.multi_search(Gs, table_capacity=1 << 22, batch_target=batch)
    assert e.value.code == 1
    for G in Gs:
        G.close()


# ---- 7. anytime
def check_anytime(seqs, w_int, r, cstar=None):
    ph = r["phases"]
    assert ph and r["lower_bound"] == max(p["lower_bound"] for p in ph)
    gs = [p["g"] for p in ph if p["finished"]]
    assert all(a >= b for a, b in zip(gs, gs[1:])), gs
    if r["finished"]:
        assert weighted_sp_score(seqs, w_int, r["rows"]) == r["g"] == min(gs)
        assert r["lower_bound"] <= r["g"]
        assert (r["finished"] == 1) == (r["lower_bound"] == r["g"])
    if cstar is not None:
        assert all(p["lower_bound"] <= cstar for p in ph)
        assert r["lower_bound"] <= cstar
        if r["finished"]:
            assert cstar <= r["g"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
@pytest.mark.parametrize("batch", [1, 16384])
def test_anytime_small(gpu_lib, name, batch):
    seqs = CASES[name]
    storm = batch == 1 and name in REOPEN_STORM  # phase 1 is w = 2: the budget of test_gpu_weighted.py
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.anytime_search(ANYTIME, table_capacity=1 << 22, batch_target=batch, max_expansions=20000 if storm else 0)
        check_anytime(seqs, G.w_int, r, c_star(name))
        if not storm:
            assert r["finished"] == 1 and r["g"] == c_star(name)
            assert [p["weight"] for p in r["phases"]] == list(ANYTIME[:len(r["phases"])])
            # the returned alignment is now the incumbent: a further exact search proves it at once
            again = G.search(table_capacity=1 << 22, batch_target=16384)
            assert again["finished"] == 2 and again["g"] == again["lower_bound"] == c_star(name)


@pytest.mark.gpu
def test_anytime_kinase(gpu_lib):
    seqs = CASES["kinase"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.anytime_search(ANYTIME, table_capacity=1 << 27, batch_target=16384)
        check_anytime(seqs, G.w_int, r, KINASE_OPT)
        assert r["finished"] == 1 and r["g"] == r["lower_bound"] == KINASE_OPT
        G.search_set_incumbent(None)
        b = G.anytime_search(ANYTIME, table_capacity=1 << 27, batch_target=16384, max_expansions=50000)
        check_anytime(seqs, G.w_int, b, KINASE_OPT)
        assert b["expansions"] <= 50000 + 16384 * 16  # a budget is checked between groups of rounds


@pytest.mark.gpu
def test_anytime_family(gpu_lib):
    """FAMILY at FAMILY_CAP coordinates, where exact search from scratch runs out of table: every phase keeps its bound, a
    proved run has lower bound == g, and a run whose exact phase runs out of table returns the best alignment with its gap.
    Measured on one B200: the exact phase runs out of table; w = 1.25 gives g = 835 366, lower bound 755 359 (g / LB 1.106)."""
    seqs = FAMILY()
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.anytime_search(ANYTIME, table_capacity=FAMILY_CAP, batch_target=16384)
        check_anytime(seqs, G.w_int, r)
        assert r["finished"] in (1, 2)
        if r["finished"] == 2:  # a phase ran out of table: the alignment of the phases before it, with its gap
            assert "table is full" in G.L.pg_last_error(G.h).decode()
            assert len(r["phases"]) < len(ANYTIME) and r["lower_bound"] < r["g"]


@pytest.mark.gpu
def test_anytime_errors(gpu_lib):
    with gpu_lib.PastarGPU(CASES["PF08184"]) as G:
        G.build_pair_tables()
        for ws in ((), (0.5,), (2, 17)):
            with pytest.raises((gpu_lib.PastarError, ValueError)) as e:
                G.anytime_search(ws)
            if isinstance(e.value, gpu_lib.PastarError):
                assert e.value.code == 1


# ---- 8. CLI
def _cli(args):
    return subprocess.run([BIN] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)


def _fasta(path, rows):
    path.write_text("".join(">s%d\n%s\n" % (i, s) for i, s in enumerate(rows)))
    return str(path)


def test_cli_incumbent_and_anytime_argument_errors(tmp_path):
    seqs = ["ACDE", "ACDF", "ACEE"]
    fa = _fasta(tmp_path / "x.fasta", seqs)
    for a in (["--anytime", "0.5"], ["--anytime", "2,,1"], ["--anytime", "abc"], ["--anytime", "2,17"], ["--anytime", "2,"],
              ["--anytime", "2,1", "--weight", "2"], ["--anytime", "2,1", "-g", "2"]):
        r = _cli(a + [fa])
        assert r.returncode == 1 and "Invalid argument" in r.stderr.decode(), (a, r.returncode, r.stderr.decode())
    bad = {
        "missing": None,
        "count": ["ACDE", "ACDF"],
        "length": ["ACDE", "ACDF-", "ACEE"],
        "residue": ["ACDE", "ACDY", "ACEE"],
        "gaps": ["ACDE-", "ACDF-", "ACEE-"],
    }
    for what, rows in bad.items():
        inc = str(tmp_path / "missing.fasta") if rows is None else _fasta(tmp_path / ("inc_%s.fasta" % what), rows)
        r = _cli(["--incumbent", inc, fa])
        assert r.returncode == 1 and "Fatal error: --incumbent" in r.stderr.decode(), (what, r.returncode, r.stderr.decode())
    for flag in ("--incumbent", "--anytime"):
        assert flag in _cli([]).stdout.decode()


def _parse(out, n):
    lines = out.split("\n")
    i = next(k for k, l in enumerate(lines) if l.startswith("Final Score:"))
    g = int(lines[i].split("g - ")[1].split(" ")[0])
    assert lines[i + 1].startswith("Lower bound: ")
    lb = int(lines[i + 1].split()[2])
    phases = [l for l in lines if l.startswith("Anytime phase ")]
    k = next(k for k, l in enumerate(lines) if l.startswith("Similarity:"))
    rows = lines[k + 2:k + 2 + n]
    return g, lb, phases, rows


@pytest.mark.gpu
def test_cli_incumbent_and_anytime_kinase(gpu_lib, tmp_path):
    seqs = CASES["kinase"]
    fa = _fasta(tmp_path / "kinase.fasta", seqs)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        opt = exact_rows(G, cap=1 << 27)["rows"]
        w_int = G.w_int
    inc = _fasta(tmp_path / "opt.fasta", opt)
    js = tmp_path / "m.json"
    r = _cli(["--incumbent", inc, "--table_capacity", "134217728", "--metrics_json", str(js), fa])
    assert r.returncode == 0, r.stderr.decode()
    g, lb, phases, rows = _parse(r.stdout.decode(), len(seqs))
    assert g == lb == KINASE_OPT and not phases
    assert "Lower bound: 421546" in r.stdout.decode()
    assert rows == opt
    d = json.load(open(js))
    assert d["incumbent"] == d["lower_bound"] == d["g"] == KINASE_OPT and d["finished"] == 2 and "phases" not in d
    r = _cli(["--anytime", "2,1", "--table_capacity", "134217728", "--metrics_json", str(js), fa])
    assert r.returncode == 0, r.stderr.decode()
    g, lb, phases, rows = _parse(r.stdout.decode(), len(seqs))
    assert g == lb == KINASE_OPT
    assert weighted_sp_score(seqs, w_int, rows) == g
    assert phases[0].startswith("Anytime phase 1: weight 2, score ") and len(phases) == 2
    assert phases[1].startswith("Anytime phase 2: weight 1, score %d, lower bound %d" % (KINASE_OPT, KINASE_OPT))
    d = json.load(open(js))
    assert d["finished"] == 1 and d["lower_bound"] == KINASE_OPT and "incumbent" not in d
    assert [p["weight"] for p in d["phases"]] == [2, 1] and d["phases"][1]["g"] == KINASE_OPT
