"""Expected values of the comparisons with the original project (test_oracle_vs_ref, test_cpp_host_cpu, test_host).

Where the original's build (oracle/_ref/pastar_ref, the unmodified sources compiled by `make -C oracle ref`) is present,
every value is computed from it live.  Elsewhere the same values come from tests/golden/ref_comparisons.json.gz, keyed
by the call and its arguments; a call the file does not hold fails.  Tables, successor records and program output are
stored as digests of their bytes (the first 64 bits of SHA-256), weights as float32 bit patterns.

Regenerate the file with the comparisons themselves:
    PG_REFDATA_RECORD=reference python -m pytest tests/test_oracle_vs_ref.py tests/test_cpp_host_cpu.py tests/test_host.py
PG_REFDATA_RECORD=project records from the components these tests pin instead (C oracle, host weights, the host
mirror's printer and reader).  The stored file was made that way, from code unchanged since its comparisons against
the original's build passed on these same inputs; the two weight routines (oracle and pg_host_weights) are checked
against each other while recording.
"""
import atexit
import gzip
import hashlib
import json
import os

import numpy as np

from conftest import GOLDEN
from oracle import oracle as O
from oracle import refio as R

PATH = os.path.join(GOLDEN, "ref_comparisons.json.gz")
RECORD = os.environ.get("PG_REFDATA_RECORD")  # None, "reference" or "project"
if RECORD == "reference":
    assert R.available(), "PG_REFDATA_RECORD=reference needs oracle/_ref/pastar_ref"
_recorded, _stored = {}, None


def digest(b):
    """First 64 bits (hex) of the SHA-256 of bytes or of an array's contiguous bytes."""
    if not isinstance(b, (bytes, bytearray)):
        b = np.ascontiguousarray(b).tobytes()
    return hashlib.sha256(b).hexdigest()[:16]


def live():
    """True where the expected values are computed by the original's build."""
    return R.available() and RECORD != "project"


def _save():
    data = {}
    if os.path.exists(PATH):
        with gzip.open(PATH, "rt") as f:
            data = json.load(f)
    data.update(_recorded)
    with gzip.GzipFile(PATH, "wb", 9, mtime=0) as f:
        f.write(json.dumps(data, separators=(",", ":"), sort_keys=True).encode())


if RECORD:
    atexit.register(_save)


def _get(fn, args, from_reference, from_project):
    key = fn + "/" + digest(repr(args).encode())
    if RECORD or R.available():
        val = json.loads(json.dumps(from_project() if RECORD == "project" else from_reference()))
        if RECORD:
            _recorded[key] = val
        return val
    global _stored
    if _stored is None:
        with gzip.open(PATH, "rt") as f:
            _stored = json.load(f)
    assert key in _stored, "%s%r: not in %s (regenerate it, see tests/refdata.py)" % (fn, args, PATH)
    return _stored[key]


def _dump_of(cost, weights, tables):
    return {"cost": digest(np.asarray(cost, dtype=np.int32)),
            "weights": np.asarray(weights, dtype=np.float32).view(np.uint32).ravel().tolist(),
            "tables": [digest(np.asarray(t, dtype=np.int32)) for t in tables], "shapes": [list(t.shape) for t in tables]}


def dump(seqs):
    """Cost table digest, weights (n * n uint32 bit patterns) and the digest and shape of every pairwise table, in the
    pair order (0,1), (0,2), ..."""
    def project():
        import mpi_pastar_msa_b200 as m
        w = O.weights(seqs)
        assert np.array_equal(w.view(np.uint32), m.host_weights(seqs).view(np.uint32))
        n = len(seqs)
        return _dump_of(O.cost_table(), w, [O.pair_table(seqs[i], seqs[j]) for i in range(n - 1) for j in range(i + 1, n)])

    def reference():
        d = R.dump(seqs)
        return _dump_of(d["cost"], d["weights"], d["tables"])
    return _get("dump", (list(seqs),), reference, project)


def _neigh_of(fpar, recs, n):
    return {"fpar": [int(f) for f in fpar], "count": [len(r) for r in recs],
            "records": [digest(np.asarray(r, dtype=O.succ_dtype(n))) for r in recs]}


def neigh(seqs, pos, g, par, vs, ht, sh):
    """Node<N>::getNeigh per parent: f of the parent, successor count, digest of the successor records."""
    n = len(seqs)

    def project():
        P = O.Problem(seqs)
        recs = [P.get_neigh(pos[k], g[k], par[k], vs, ht, sh) for k in range(len(pos))]
        return _neigh_of([int(g[k]) + P.calculate_h(pos[k]) for k in range(len(pos))], recs, n)

    def reference():
        res = R.neigh(seqs, pos, g, par, vs, ht, sh)
        return _neigh_of([r[0] for r in res], [r[1] for r in res], n)
    args = (list(seqs), np.asarray(pos).tolist(), np.asarray(g).tolist(), np.asarray(par).tolist(), vs, ht, sh)
    return _get("neigh", args, reference, project)


def astar(seqs):
    """Serial A*: [optimal g, expansions, generated]."""
    def project():
        a = O.Problem(seqs).astar(want_rows=False)
        return [a["g"], a["expansions"], a["generated"]]

    def reference():
        r = R.astar(seqs)
        return [r["g"], r["expansions"], r["generated"]]
    return _get("astar", (list(seqs),), reference, project)


def program_output(what, args, ref_run, project_run):
    """[return code, digest of stdout] of the original's program; ref_run / project_run return (rc, stdout bytes)."""
    def wrap(run):
        rc, out = run()
        return [rc, digest(out)]
    return _get(what, args, lambda: wrap(ref_run), lambda: wrap(project_run))
