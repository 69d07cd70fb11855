"""Incumbent-bounded and anytime search on one GPU: python tools/anytime_sweep.py

For each input (kinase; FAMILY, the family that exact search cannot finish in 2^22 coordinates; fam7x30 and fam5x60,
also at one parent per round; S7 under an expansion budget) it prints one JSON line per run:
  - "exact": the unbounded exact search;
  - "exact_inc_w2": exact search with the w = 2 alignment as incumbent (U = its cost);
  - "exact_inc_opt": exact search with an optimal alignment as incumbent (U = C*), when one is known from another run;
  - "anytime": the default schedule (2, 1.25, 1) from no incumbent, with its phases.
Each line has finished, g, the certified lower bound, inserted (distinct coordinates stored), probed (table lookups),
expansions, kernel_ms (device time of the search rounds) and the GPU's name and power limit.  A run that fails
(PG_ERR_CAPACITY) prints its error.  profiles/r04_anytime_sweep.json is this output on a B200."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mpi_pastar_msa_b200 as m  # noqa: E402
from conftest import CASES, S7, family_seqs  # noqa: E402

INPUTS = [  # name, sequences, table capacity (coordinates), expansion budget of every run, batches
    ("kinase", CASES["kinase"], 1 << 27, 0, [16384]),
    ("family_seqs(8,150,105,0.2,0.04)", family_seqs(8, 150, 105, 0.2, 0.04), 1 << 22, 0, [16384]),
    ("fam7x30", CASES["fam7x30"], 1 << 22, 0, [1, 16384]),
    ("fam5x60", CASES["fam5x60"], 1 << 22, 0, [1]),
    ("S7", S7(), 1 << 26, 2_000_000, [16384]),
]
KEYS = ("finished", "g", "lower_bound", "inserted", "probed", "expansions", "pushed", "reopen", "kernel_ms")


def run(G, line, **kw):
    try:
        r = G.search(**kw)
    except m.PastarError as e:
        line.update({"finished": 0, "error": str(e)})
        return None
    line.update({k: r[k] for k in KEYS})
    return r


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         universal_newlines=True).stdout.strip()
    for name, seqs, cap, budget, batches in INPUTS:
        with m.PastarGPU(seqs) as G:
            G.build_pair_tables()
            for batch in batches:
                base = {"input": name, "table_capacity": cap, "max_expansions": budget, "batch": batch, "gpu": gpu}
                opt_rows = None
                G.search_set_weight(1, 1)
                G.search_set_incumbent(None)
                line = dict(base, run="exact")
                r = run(G, line, table_capacity=cap, batch_target=batch, max_expansions=budget)
                print(json.dumps(line), flush=True)
                if r and r["finished"] == 1:
                    opt_rows = r["rows"]
                # the w = 2 alignment at batch 16384 (one parent per round reopens heavily at w = 2 on some inputs)
                w2 = G.search(table_capacity=cap, batch_target=16384, max_expansions=budget, weight=2)
                G.search_set_weight(1, 1)
                w2_rows = w2["rows"] if w2["finished"] else None
                line = dict(base, run="anytime", weights=[2, 1.25, 1])
                try:
                    a = G.anytime_search((2, 1.25, 1), table_capacity=cap, batch_target=batch, max_expansions=budget)
                    line.update({k: a[k] for k in KEYS})
                    line["phases"] = a["phases"]
                    if len(a["phases"]) < 3 and a["lower_bound"] < a["g"]:  # stopped by the table or the budget
                        line["stopped"] = G.L.pg_last_error(G.h).decode()
                    if a["finished"] == 1 and opt_rows is None:
                        opt_rows = a["rows"]
                except m.PastarError as e:
                    line.update({"finished": 0, "error": str(e)})
                print(json.dumps(line), flush=True)
                for tag, rows in (("exact_inc_w2", w2_rows), ("exact_inc_opt", opt_rows)):
                    if rows is None:
                        continue
                    G.search_set_incumbent(rows)
                    line = dict(base, run=tag, incumbent=G.score_alignment(rows))
                    run(G, line, table_capacity=cap, batch_target=batch, max_expansions=budget, want_rows=False)
                    print(json.dumps(line), flush=True)
                G.search_set_incumbent(None)


if __name__ == "__main__":
    main()
