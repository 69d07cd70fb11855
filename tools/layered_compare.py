"""Layered search against A* on one GPU: cost or final bound, passes, levels, expansions, the coordinates held and the
time, beside pg_search's inserted, expansions and kernel time.

    python tools/layered_compare.py [--out profiles/r05_layered.json] [--cap 4194304] [--budget 300000000] [names...]

Inputs: kinase, fam5x60, fam7x30, fam10x100 and FAMILY (family_seqs(8, 150, 105, 0.2, 0.04)).  The layered search runs at
--cap coordinates and --budget expansions over all its passes; A* runs at batch 16384 with a 2^27 table (FAMILY: 2^22,
where it runs out of table)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import CASES, WIDE_CASES, family_seqs  # noqa: E402

import mpi_pastar_msa_b200 as m  # noqa: E402

INPUTS = {"kinase": CASES["kinase"], "fam5x60": CASES["fam5x60"], "fam7x30": CASES["fam7x30"],
          "fam10x100": WIDE_CASES["fam10x100"], "FAMILY": family_seqs(8, 150, 105, 0.2, 0.04)}


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                              timeout=30).stdout.decode().strip()
    except Exception as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_layered.json"))
    ap.add_argument("--cap", type=int, default=1 << 22)
    ap.add_argument("--budget", type=int, default=300_000_000)
    ap.add_argument("names", nargs="*")
    a = ap.parse_args()
    out = {"gpu": gpu_info(), "table_capacity": a.cap, "max_expansions": a.budget, "inputs": {}}
    for name in a.names or list(INPUTS):
        seqs = INPUTS[name]
        row = {}
        with m.PastarGPU(seqs) as G:
            G.build_pair_tables()
            t = time.time()
            try:
                r = G.layered_search(table_capacity=a.cap, max_expansions=a.budget)
                st = r["layered"]
                row["layered"] = {"finished": r["finished"], "g": r["g"], "lower_bound": r["lower_bound"],
                                  "iterations": st["iterations"], "first_bound": st["first_bound"], "last_bound": st["last_bound"],
                                  "passes": st["passes"], "levels": st["levels"], "depth": st["depth"],
                                  "top_expansions": st["top_expansions"], "expansions": r["expansions"],
                                  "inserted": r["inserted"], "max_level_nodes": st["max_level_nodes"], "max_held": st["max_held"],
                                  "peak_bytes": st["peak_bytes"], "kernel_ms": round(r["kernel_ms"], 2),
                                  "wall_s": round(time.time() - t, 3)}
            except m.PastarError as e:
                row["layered"] = {"error": str(e), "wall_s": round(time.time() - t, 3)}
            m.release_cached_memory()
            cap = 1 << 22 if name == "FAMILY" else 1 << 27
            t = time.time()
            try:
                r = G.search(table_capacity=cap, batch_target=16384, want_rows=False)
                row["astar"] = {"table_capacity": cap, "finished": r["finished"], "g": r["g"], "inserted": r["inserted"],
                                "expansions": r["expansions"], "kernel_ms": round(r["kernel_ms"], 2),
                                "wall_s": round(time.time() - t, 3)}
            except m.PastarError as e:
                row["astar"] = {"table_capacity": cap, "error": str(e), "wall_s": round(time.time() - t, 3)}
            m.release_cached_memory()
        out["inputs"][name] = row
        print(name, json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
