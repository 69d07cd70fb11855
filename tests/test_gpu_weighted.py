"""Bounded-suboptimal (weighted) search: f_w = g + h_w orders the open list, the returned alignment costs at most w x the
optimum, and pg_search_lower_bound certifies it (LB <= C* <= g, g * den <= num * LB).  Weight 1 is the exact search."""
import functools
import os
import subprocess

import numpy as np
import pytest

from conftest import CASES, KNOWN_OPT, ROOT, WIDE_CASES, family_seqs, random_parents, weighted_sp_score
from oracle import oracle as O

INT_MAX = 2**31 - 1
SMALL = ["test", "test2", "PF08184", "rnd4x60", "fam6x80", "fam3x300", "fam5x60", "fam4x150", "fam7x30", "fam8x20"]
KINASE_H0 = 408457  # h(start) of kinase, SURVEY section 4
# a family that exact search cannot finish in FAMILY_CAP coordinates (see test_weighted_reaches_what_exact_cannot)
FAMILY = lambda: family_seqs(8, 150, 105, 0.2, 0.04)
FAMILY_CAP = 1 << 22
BIN = os.path.join(ROOT, "mpi_pastar_msa_b200", "bin", "pastar")


@functools.lru_cache(maxsize=None)
def c_star(name):
    return KNOWN_OPT.get(name) or O.Problem(CASES[name]).astar(want_rows=False)["g"]


def check_bound(seqs, w_int, r, cstar):
    """finished, rows spell the sequences and re-score to g, LB <= C* <= g <= w * LB."""
    assert r["finished"] == 1, r
    assert weighted_sp_score(seqs, w_int, r["rows"]) == r["g"] == r["f"]
    assert r["lower_bound"] <= cstar <= r["g"], (r["lower_bound"], cstar, r["g"])
    assert r["g"] * r["weight_den"] <= r["weight_num"] * r["lower_bound"], r


# ---- 1. weight 1 is today's search
@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
@pytest.mark.parametrize("batch", [1, 16384])
def test_weight_one_is_exact_search(gpu_lib, name, batch):
    seqs = CASES[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        a = G.search(table_capacity=1 << 22, batch_target=batch)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        G.search_set_weight(1, 1)
        b = G.search(table_capacity=1 << 22, batch_target=batch)
    assert a["finished"] == b["finished"] == 1
    assert a["g"] == b["g"] == c_star(name)
    if batch == 1:  # one parent per round: the search is deterministic
        assert a["rows"] == b["rows"]
        for k in ("expansions", "generated", "pushed", "reopen"):
            assert a[k] == b[k], k
    else:  # successors of one round race for equal-g ties, so the optimal alignment returned may differ between runs
        assert weighted_sp_score(seqs, G.w_int, a["rows"]) == weighted_sp_score(seqs, G.w_int, b["rows"]) == a["g"]
    assert a["lower_bound"] == a["g"] and b["lower_bound"] == b["g"]


# ---- 2. the bound holds
# One parent per round and w >= 2 on these two inputs: the weighted best-first order keeps reaching nodes by expensive
# paths and then improving them - measured on a B200 at 300 000 expansions, still unfinished, with 270 000 (rnd4x60) and
# 220 000 - 250 000 (fam7x30) reopenings (exact search: 79 and 4 014 expansions).  They run under an expansion budget
# and check the bound a budgeted run reports; at batch 16384 and at w = 1.25 they run to the end.
REOPEN_STORM = {"rnd4x60", "fam7x30"}


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
@pytest.mark.parametrize("weight", [1.25, 2, 4])
@pytest.mark.parametrize("batch", [1, 16384])
def test_weighted_bound_small(gpu_lib, name, weight, batch):
    seqs = CASES[name]
    storm = batch == 1 and weight >= 2 and name in REOPEN_STORM
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        h0 = int(G.calculate_h(np.zeros((1, len(seqs)), dtype=np.uint16))[0])
        r = G.search(table_capacity=1 << 22, batch_target=batch, weight=weight, max_expansions=20000 if storm else 0)
        assert (r["weight_num"], r["weight_den"]) == gpu_lib.weight_fraction(weight)
        if storm:
            assert r["finished"] == 0 and h0 <= r["lower_bound"] <= c_star(name)
        else:
            check_bound(seqs, G.w_int, r, c_star(name))


# ---- 3. kinase
@pytest.mark.gpu
def test_weighted_kinase(gpu_lib):
    seqs = CASES["kinase"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        exact = G.search(table_capacity=1 << 27, batch_target=16384, want_rows=False)
        assert exact["g"] == exact["lower_bound"] == 421546
        for w in (1.5, 2):
            r = G.search(table_capacity=1 << 27, batch_target=16384, weight=w)
            check_bound(seqs, G.w_int, r, 421546)
            assert r["expansions"] < exact["expansions"], (w, r["expansions"], exact["expansions"])


# ---- 4. reaches what exact search cannot
@pytest.mark.gpu
def test_weighted_reaches_what_exact_cannot(gpu_lib):
    """FAMILY = family_seqs(8, 150, 105, 0.2, 0.04) at FAMILY_CAP = 2^22 coordinates, batch 16384.  Exact search runs out
    of table (PG_ERR_CAPACITY) or hits the 3 M-expansion budget; w = 2 finishes.  Measured on a B200: exact search
    PG_ERR_CAPACITY; w = 2 g = 843 195, lower bound 755 204 (g / LB = 1.117), 650 expansions (profiles/r03_weighted_sweep.json)."""
    seqs = FAMILY()
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        try:
            r1 = G.search(table_capacity=FAMILY_CAP, batch_target=16384, max_expansions=3_000_000, want_rows=False)
            assert r1["finished"] == 0, r1
        except gpu_lib.PastarError as e:
            assert e.code == 4  # PG_ERR_CAPACITY
        r = G.search(table_capacity=FAMILY_CAP, batch_target=16384, weight=2)
        assert r["finished"] == 1
        assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"]
        assert r["g"] * r["weight_den"] <= r["weight_num"] * r["lower_bound"]


# ---- 5. wide key / wide value
@pytest.mark.gpu
def test_weighted_wide_key(gpu_lib):
    seqs = WIDE_CASES["fam10x100"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.search(table_capacity=1 << 24, batch_target=4096, weight=2)
        check_bound(seqs, G.w_int, r, KNOWN_OPT["fam10x100"])


@pytest.mark.gpu
def test_weighted_wide_value(gpu_lib, monkeypatch):
    monkeypatch.setenv("PG_VALW", "8")
    seqs = CASES["fam6x80"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        r = G.search(table_capacity=1 << 22, batch_target=1024, weight=2)
        check_bound(seqs, G.w_int, r, c_star("fam6x80"))


# ---- 6. partitioned
@pytest.mark.gpu
@pytest.mark.parametrize("name,parts,batch,ht,sh", [("fam5x60", 2, 256, "FZORDER", 0), ("fam8x20", 4, 4096, "PZORDER", 1)])
def test_weighted_multi_search(gpu_lib, name, parts, batch, ht, sh):
    seqs = CASES[name]
    Gs = []
    for _ in range(parts):
        G = gpu_lib.PastarGPU(seqs)
        G.build_pair_tables()
        G.configure_hash(ht, sh)
        Gs.append(G)
    tot, _ = gpu_lib.multi_search(Gs, table_capacity=1 << 22, batch_target=batch, weight=2)
    check_bound(seqs, Gs[0].w_int, tot, c_star(name))
    assert all(G.search_lower_bound() == tot["lower_bound"] for G in Gs)
    for G in Gs:
        G.close()


def partitioned_search(m, seqs, parts, batch, hash_type, shift, weight, cap=1 << 22):
    """The loop-back step-wise driver of test_gpu_partitioned.py (outbox device pointers handed to the owners' inserts),
    weighted; returns the best goal, the backtraced rows and the minimum of the partitions' lower bounds."""
    Gs = []
    for r in range(parts):
        G = m.PastarGPU(seqs)
        G.build_pair_tables()
        G.configure_hash(hash_type, shift)
        G.search_set_weight(*m.weight_fraction(weight))
        G.search_begin(parts, r, cap, batch)
        Gs.append(G)
    best, rounds = INT_MAX, 0
    while True:
        for G in Gs:
            G.search_round(best)
        boxes = [[G.search_outbox(d) if d != r else (0, 0) for d in range(parts)] for r, G in enumerate(Gs)]
        for r in range(parts):
            for d in range(parts):
                ptr, n = boxes[r][d]
                if n:
                    Gs[d].search_insert_dev(ptr, n)
        st = [G.search_status() for G in Gs]
        mn = min(s[0] for s in st)
        best = min(s[1] for s in st)
        rounds += 1
        assert rounds < 200000
        if mn >= best or mn == INT_MAX:
            break
    res = {"g": best, "lower_bound": min(G.search_lower_bound() for G in Gs)}
    n = len(seqs)
    pos = [len(s) for s in seqs]
    cols = []
    while any(pos):
        own = int(Gs[0].owner(np.array(pos, dtype=np.uint16), parts)[0])
        hit = Gs[own].search_lookup(pos)
        assert hit is not None, pos
        cols.append(hit[1])
        pos = [p - ((hit[1] >> i) & 1) for i, p in enumerate(pos)]
    rows, at = [[] for _ in range(n)], [0] * n
    for mask in reversed(cols):
        for i in range(n):
            if (mask >> i) & 1:
                rows[i].append(seqs[i][at[i]])
                at[i] += 1
            else:
                rows[i].append("-")
    res["rows"] = ["".join(r) for r in rows]
    for G in Gs:
        G.search_end()
        G.close()
    return res


@pytest.mark.gpu
def test_weighted_stepwise_partitioned(gpu_lib):
    """The caller's own backtrace may spell an alignment cheaper than the best goal: C* <= score <= best goal <= w LB."""
    name = "fam5x60"
    seqs = CASES[name]
    r = partitioned_search(gpu_lib, seqs, 2, 256, "FZORDER", 0, 2)
    w = gpu_lib.host_weights(seqs).astype(np.int32)
    assert c_star(name) <= weighted_sp_score(seqs, w, r["rows"]) <= r["g"] <= 2 * r["lower_bound"]


# ---- 7. budgeted runs report a valid bound
@pytest.mark.gpu
def test_budgeted_weighted_bound(gpu_lib):
    """w = 2 solves kinase in about 2 600 expansions (280 rounds), under the 100 000 budget: the bound holds either way.
    One parent per round and a 100-expansion budget stop the search short of the goal: every alignment has at least 276
    columns, and each of its nodes but the goal must be expanded first."""
    with gpu_lib.PastarGPU(CASES["kinase"]) as G:
        G.build_pair_tables()
        r = G.search(table_capacity=1 << 27, batch_target=16384, max_expansions=100000, weight=2)
        assert KINASE_H0 <= r["lower_bound"] <= 421546
        if r["finished"]:
            check_bound(CASES["kinase"], G.w_int, r, 421546)
        r = G.search(table_capacity=1 << 27, batch_target=1, max_expansions=100, weight=2, want_rows=False)
        assert r["finished"] == 0 and r["expansions"] >= 100
        assert KINASE_H0 <= r["lower_bound"] <= 421546


@pytest.mark.gpu
def test_budgeted_exact_bound_stepwise(gpu_lib):
    with gpu_lib.PastarGPU(CASES["kinase"]) as G:
        G.build_pair_tables()
        G.search_begin(1, 0, 1 << 27, 16384)
        while True:
            G.search_round()
            mn, best, cnt = G.search_status()
            if cnt["expansions"] >= 100000:
                break
        lb = G.search_lower_bound()
        assert best == INT_MAX or best > mn
        assert KINASE_H0 <= mn <= lb <= 421546, (mn, lb)
        G.search_end()


# ---- 8. getNeigh stays unweighted
@pytest.mark.gpu
def test_expand_batch_ignores_weight(gpu_lib):
    seqs = CASES["fam6x80"]
    pos, g, par = random_parents(seqs, 300, 7)
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        nodes = G.make_nodes(pos, g, par)
        a, ca = G.expand_batch(nodes, 4)
        h = G.calculate_h(pos)
        G.search_set_weight(2, 1)
        b, cb = G.expand_batch(nodes, 4)
        assert np.array_equal(ca, cb) and a.tobytes() == b.tobytes()
        assert np.array_equal(G.calculate_h(pos), h)


# ---- 9. errors
@pytest.mark.gpu
def test_weight_errors(gpu_lib):
    seqs = CASES["PF08184"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        with pytest.raises(gpu_lib.PastarError) as e:
            G.search_lower_bound()
        assert e.value.code == 5  # no search yet
        for num, den in ((1, 2), (3, 3), (2, 0), (17, 1), (16 * 1024 + 1, 1024), (4096, 2048)):
            with pytest.raises(gpu_lib.PastarError) as e:
                G.search_set_weight(num, den)
            assert e.value.code == 1, (num, den)
        G.search_begin(1, 0, 1 << 20, 256)
        with pytest.raises(gpu_lib.PastarError) as e:
            G.search_set_weight(2, 1)
        assert e.value.code == 5  # PG_ERR_STATE
        G.search_end()
        G.search_set_weight(2, 1)
    a, b = gpu_lib.PastarGPU(seqs), gpu_lib.PastarGPU(seqs)
    for G in (a, b):
        G.build_pair_tables()
    a.search_set_weight(2, 1)
    with pytest.raises(gpu_lib.PastarError) as e:
        gpu_lib.multi_search([a, b], table_capacity=1 << 20, batch_target=256)
    assert e.value.code == 1
    a.close()
    b.close()


@pytest.mark.gpu
def test_weighted_range_unsupported(gpu_lib):
    """All pair weights K: UB and h(start) scale with K, so K is chosen for an exact f range below 2^27 buckets and a
    weight-16 range above it.  UB is the cost of the all-advance alignment (every sequence padded with trailing gaps)."""
    seqs = CASES["fam4x150"]
    n, L = len(seqs), max(len(s) for s in seqs)
    ones = np.ones((n, n), dtype=np.int32)
    ub1 = weighted_sp_score(seqs, ones, [s + "-" * (L - len(s)) for s in seqs])
    with gpu_lib.PastarGPU(seqs, weights=ones) as G:
        G.build_pair_tables()
        h01 = int(G.calculate_h(np.zeros((1, n), dtype=np.uint16))[0])
    K = (1 << 27) // (16 * ub1 - h01) + 1
    assert K * (ub1 - h01) + 2 <= 1 << 27 < K * (16 * ub1 - h01) + 2 and 16 * K * ub1 < INT_MAX
    with gpu_lib.PastarGPU(seqs, weights=ones * K) as G:
        G.build_pair_tables()
        G.search_begin(1, 0, 1 << 20, 256)
        G.search_end()
        G.search_set_weight(16, 1)
        with pytest.raises(gpu_lib.PastarError) as e:
            G.search_begin(1, 0, 1 << 20, 256)
        assert e.value.code == 3  # PG_ERR_UNSUPPORTED


# ---- 10. CLI, no device
def _cli(args):
    return subprocess.run([BIN] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)


def test_cli_weight_argument_errors(tmp_path):
    fa = tmp_path / "x.fasta"
    fa.write_text(">a\nACDE\n>b\nACDF\n>c\nACEE\n")
    for w in ("0.5", "abc", "17", "2x", "nan"):
        r = _cli(["--weight", w, str(fa)])
        assert r.returncode == 1 and "Invalid argument" in r.stderr.decode(), (w, r.returncode, r.stderr.decode())
    # a prefix of --weight is accepted: the run gets past the parser and stops at the missing file
    r = _cli(["--wei", "2", str(tmp_path / "missing.fasta")])
    assert r.returncode == 1 and "is not a regular file." in r.stdout.decode()
    assert "Invalid argument" not in r.stderr.decode()
    assert "--weight" in _cli([]).stdout.decode()


@pytest.mark.gpu
def test_cli_weighted_kinase(tmp_path):
    import json
    import mpi_pastar_msa_b200 as m
    seqs = CASES["kinase"]
    fa, js = tmp_path / "kinase.fasta", tmp_path / "m.json"
    fa.write_text("".join(">s%d\n%s\n" % (i, s) for i, s in enumerate(seqs)))
    r = _cli(["--weight", "2", "--table_capacity", "134217728", "--metrics_json", str(js), str(fa)])
    assert r.returncode == 0, r.stderr.decode()
    lines = r.stdout.decode().split("\n")
    i = next(k for k, l in enumerate(lines) if l.startswith("Final Score:"))
    g = int(lines[i].split("g - ")[1].split(" ")[0])
    assert lines[i + 1].startswith("Lower bound: ")
    lb = int(lines[i + 1].split()[2])
    rows = lines[i + 5:i + 5 + len(seqs)]
    assert weighted_sp_score(seqs, m.host_weights(seqs).astype("int32"), rows) == g
    assert lb <= 421546 <= g <= 2 * lb
    d = json.load(open(js))
    assert d["weight"] == 2 and d["lower_bound"] == lb and d["g"] == g
