"""Beam search (pg_search_beam) on one GPU: one single-width run per input and width, and kinase's layered search with and
without the beam's alignment as its incumbent.

    python tools/beam_sweep.py [--out profiles/r06_beam.json] [names...]

Inputs: kinase, fam7x30, fam10x100, FAMILY (family_seqs(8, 150, 105, 0.2, 0.04)) and S7 (random_seqs(7, 500, 12345)).
Widths 2^10, 2^14 and 2^18, and 2^20 for FAMILY, each at the default table capacity.  Per run: g, the certified lower bound,
g / C* where C* is known, device ms (CUDA events around the whole run), ms per level, peak device bytes, levels, nodes kept
and dropped, and the most candidates of one level before the cut (also over W)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import CASES, KNOWN_OPT, S7, WIDE_CASES, family_seqs  # noqa: E402

import mpi_pastar_msa_b200 as m  # noqa: E402

INPUTS = {"kinase": CASES["kinase"], "fam7x30": CASES["fam7x30"], "fam10x100": WIDE_CASES["fam10x100"],
          "FAMILY": family_seqs(8, 150, 105, 0.2, 0.04), "S7": S7()}
WIDTHS = [1 << 10, 1 << 14, 1 << 18]
EXTRA = {"FAMILY": [1 << 20]}


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                              timeout=30).stdout.decode().strip()
    except Exception as e:
        return "unknown (%s)" % e


def optimum(name):
    if name in KNOWN_OPT:
        return KNOWN_OPT[name]
    if name == "fam7x30":
        from oracle import oracle as O
        return O.Problem(INPUTS[name]).astar(want_rows=False)["g"]
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_beam.json"))
    ap.add_argument("names", nargs="*")
    a = ap.parse_args()
    out = {"gpu": gpu_info(), "inputs": {}}
    for name in a.names or list(INPUTS):
        seqs = INPUTS[name]
        cstar = optimum(name)
        row = {"C*": cstar, "runs": []}
        with m.PastarGPU(seqs) as G:
            G.build_pair_tables()
            G.beam_search([16], want_rows=False)  # warm-up: module load, first launches
            G.search_set_incumbent(None)          # its alignment would bound the first width
            for W in WIDTHS + EXTRA.get(name, []):
                t = time.time()
                try:
                    r = G.beam_search([W])
                    st = r["beam"]
                    run = {"width": W, "finished": r["finished"], "g": r["g"], "lower_bound": r["lower_bound"],
                           "g_over_cstar": round(r["g"] / cstar, 5) if cstar and r["g"] > 0 else None,
                           "kernel_ms": round(r["kernel_ms"], 2), "ms_per_level": round(r["kernel_ms"] / max(1, st["levels"]), 4),
                           "peak_bytes": st["peak_bytes"], "levels": st["levels"], "kept": st["kept"], "dropped": st["dropped"],
                           "max_candidates": st["max_candidates"], "max_candidates_over_width": round(st["max_candidates"] / W, 3),
                           "retained": st["retained"], "expansions": r["expansions"], "wall_s": round(time.time() - t, 3)}
                    if W == WIDTHS[-1] and r["finished"]:
                        row["rows_at_%d" % W] = r["rows"]
                except m.PastarError as e:
                    run = {"width": W, "error": str(e), "wall_s": round(time.time() - t, 3)}
                G.search_set_incumbent(None)
                m.release_cached_memory()
                row["runs"].append(run)
                print(name, json.dumps(run), flush=True)
            if name == "kinase":
                inc = row.pop("rows_at_%d" % WIDTHS[-1], None)
                lay = {}
                for label, rows in (("without_incumbent", None), ("beam_incumbent", inc)):
                    G.search_set_incumbent(None)
                    r = G.layered_search(incumbent=rows, table_capacity=1 << 22)
                    st = r["layered"]
                    lay[label] = {"incumbent": G.score_alignment(rows) if rows else None, "finished": r["finished"], "g": r["g"],
                                  "iterations": st["iterations"], "passes": st["passes"], "first_bound": st["first_bound"],
                                  "last_bound": st["last_bound"], "expansions": r["expansions"],
                                  "kernel_ms": round(r["kernel_ms"], 2)}
                    print(name, label, json.dumps(lay[label]), flush=True)
                    m.release_cached_memory()
                G.search_set_incumbent(None)
                row["layered"] = lay
            row.pop("rows_at_%d" % WIDTHS[-1], None)
        out["inputs"][name] = row
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
