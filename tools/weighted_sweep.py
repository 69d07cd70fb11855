"""Weighted (bounded-suboptimal) search on one GPU: python tools/weighted_sweep.py [weights...]

Runs kinase and a family input that exact search cannot finish at a fixed table capacity (FAMILY below, the one
tests/test_gpu_weighted.py uses) at w = 1, 1.1, 1.25, 1.5, 2, 3 and prints one JSON line per run: w, finished, g, the
certified lower bound LB, g / LB, expansions, pops, kernel_ms (device time of the search rounds) and wall seconds (the
pg_search call).  A run that fails (PG_ERR_CAPACITY) prints its error instead.  profiles/r03_weighted_sweep.json is this
output on a B200."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mpi_pastar_msa_b200 as m  # noqa: E402
from conftest import CASES, family_seqs  # noqa: E402

INPUTS = [  # name, sequences, table capacity (coordinates), expansion budget of the run
    ("kinase", CASES["kinase"], 1 << 27, 0),
    ("family_seqs(8,150,105,0.2,0.04)", family_seqs(8, 150, 105, 0.2, 0.04), 1 << 22, 3_000_000),
]


def main():
    weights = [float(a) for a in sys.argv[1:]] or [1, 1.1, 1.25, 1.5, 2, 3]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         universal_newlines=True).stdout.strip()
    for name, seqs, cap, budget in INPUTS:
        with m.PastarGPU(seqs) as G:
            G.build_pair_tables()
            for w in weights:
                line = {"input": name, "w": w, "weight_num": m.weight_fraction(w)[0], "weight_den": m.WEIGHT_DEN,
                        "table_capacity": cap, "max_expansions": budget, "gpu": gpu}
                t0 = time.perf_counter()
                try:
                    # weight 1 is set explicitly: the context keeps the weight of the previous run otherwise
                    G.search_set_weight(*m.weight_fraction(w))
                    r = G.search(table_capacity=cap, batch_target=16384, max_expansions=budget, want_rows=False)
                except m.PastarError as e:
                    line.update({"finished": 0, "error": str(e), "wall_s": time.perf_counter() - t0})
                    print(json.dumps(line), flush=True)
                    continue
                lb = r["lower_bound"]
                line.update({"finished": r["finished"], "g": r["g"] if r["finished"] else None, "lower_bound": lb,
                             "g_over_lb": r["g"] / lb if r["finished"] else None, "expansions": r["expansions"],
                             "pops": r["pops"], "reopen": r["reopen"], "kernel_ms": r["kernel_ms"], "wall_s": r["seconds"]})
                print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
