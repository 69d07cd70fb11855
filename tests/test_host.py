"""CPU: host-side product code and the C-ABI library surface (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import CASES, GOLDEN, ROOT, S7, has_gpu

import mpi_pastar_msa_b200 as m
from mpi_pastar_msa_b200 import api

G = np.load(os.path.join(GOLDEN, "reference_golden.npz"))
ALL = dict(CASES)
ALL["S7"] = S7()


def test_library_loads_and_exports_every_declared_symbol():
    L = m.load_library()
    assert L.pg_abi_version() == 1
    hdr = open(os.path.join(ROOT, "include", "pastar_gpu.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(pg_[a-z0-9_]+)\s*\(", hdr)) - {"pg_node_stride", "pg_succ_stride"}  # static inline
    assert len(declared) >= 20
    raw = ctypes.CDLL(m.lib_path())
    for name in sorted(declared):
        assert hasattr(raw, name), name
    assert declared == set(api.EXPORTS)


def test_record_layouts_match_reference_node_sizes():
    # sizeof(Node<N>) verified against the reference (SURVEY F7)
    sizes = {3: 20, 4: 20, 5: 24, 6: 24, 7: 28, 8: 28, 9: 32, 10: 32, 14: 40, 16: 44}
    for n, sz in sizes.items():
        assert m.node_dtype(n).itemsize == sz
        assert m.succ_dtype(n).itemsize == sz + 4
        assert m.node_dtype(n).fields["f"][1] == ((2 * n + 3) & ~3)


def test_default_cost_table():
    assert np.array_equal(m.default_cost_table(), G["cost_table"])


@pytest.mark.parametrize("name", list(ALL))
def test_host_weights_bit_exact_vs_reference(name):
    """pg_host_weights (product host code) == weightAltschulsRationale2 of the reference, float bit patterns."""
    w = m.host_weights(ALL[name])
    assert np.array_equal(w.view(np.uint32), G[name + "/weights_f32"].view(np.uint32))


def test_host_weights_beyond_reference_limit():
    # the reference heap-overflows at L >= 999 (SURVEY F4); the product accepts it and stays finite and >= 8
    from conftest import random_seqs
    w = m.host_weights(random_seqs(3, 1200, 5))
    iu = np.triu_indices(3, 1)
    assert np.isfinite(w[iu]).all() and (w[iu].astype(np.int32) >= 8).all()


def test_read_fasta_rules(tmp_path):
    p = tmp_path / "x.fasta"
    p.write_text(">a\nAC\nGT\n\n>b\nTT\n>c\n>d\nGG")  # '>' and empty lines end a record; empty records are dropped
    assert m.read_fasta(str(p)) == ["ACGT", "TT", "GG"]
    for name in ("test", "test2", "PF08184", "kinase"):  # the reference fixtures, written as multi-line records
        src = tmp_path / (name + ".fasta")
        src.write_text("".join(">%s_%d\n%s\n" % (name, i, "\n".join(q[k:k + 60] for k in range(0, len(q), 60)))
                               for i, q in enumerate(CASES[name])))
        assert m.read_fasta(str(src)) == CASES[name]


@pytest.mark.skipif(has_gpu(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    with pytest.raises(m.PastarError) as e:
        m.PastarGPU(CASES["PF08184"])
    assert e.value.code == 2  # PG_ERR_CUDA


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "mpi_pastar_msa_b200")
    for d, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                src = open(os.path.join(d, f), errors="ignore").read()
                assert "pastar_oracle" not in src and "from oracle" not in src and "import oracle" not in src, f


def _weight_edge_cases():
    import random
    from conftest import family_seqs
    al = "ACDEFGHIKLMNPQRSTVWY"
    rng = random.Random(7)
    cases = {}
    for n in (3, 4, 5, 6, 7, 8, 9, 10, 14, 16):
        cases["ragged%d" % n] = ["".join(rng.choice(al) for _ in range(rng.randint(1, 90))) for _ in range(n)]
        cases["fam%d" % n] = family_seqs(n, 40 + 3 * n, 100 + n, sub=0.2, indel=0.05)
    cases["identical4"] = ["ACDEFGHIKL"] * 4            # all pair distances 0: the neighbour-joining tie path
    cases["identical3_len1"] = ["A"] * 3
    cases["len1_mixed"] = ["A", "C", "DE", "F", "GHI"]
    cases["two_groups"] = ["AAAAAAAAAA", "AAAAAAAAAC", "WWWWWWWWWW", "WWWWWWWWWY", "AAAAWWWWWW"]  # reference yields inf weights
    cases["rare_letters"] = ["ABXXJOU", "BJXBOXAA", "UOJACD", "ACDXB"]  # letters with unset PAM rows (SURVEY F2); not 'Z': index 90 is out of the reference's table (its output then varies with the environment)
    return cases


@pytest.mark.parametrize("name", list(_weight_edge_cases()))
def test_host_weights_edge_cases_vs_reference_build(name):
    """pg_host_weights against the reference compiled in place (oracle/_ref), float bit patterns, on inputs the golden
    file does not hold: ragged lengths down to 1, every supported N, identical sequences (zero distances), two distant
    groups (the reference's weights overflow to inf there, and so must ours), letters with unset PAM rows.  Without the
    build the reference's bit patterns come from tests/golden/ref_comparisons.json.gz (tests/refdata.py)."""
    import refdata
    seqs = _weight_edge_cases()[name]
    w = m.host_weights(seqs)
    assert w.view(np.uint32).ravel().tolist() == refdata.dump(seqs)["weights"]


def test_host_weights_refuses_residues_outside_the_cost_table():
    # 'Z' = index 90 reads past pam250['Z']['Z'] in the reference (Cost.h:49); refused like pg_ctx_create / pg_gpu_weights do
    with pytest.raises(api.PastarError):
        m.host_weights(["ACDZ", "ACDE", "ACD"])
    with pytest.raises(api.PastarError):
        m.host_weights(["ACDe", "ACDE", "ACD"])   # lowercase: also outside the 90 x 90 table


def test_every_entry_point_refuses_null_arguments():
    """No entry point dereferences a null context / buffer: PG_ERR_ARG (or 0 for the size getters), never a crash.  Run in a
    child process so that a crash fails this test instead of ending the session; nothing here reaches the CUDA runtime."""
    import subprocess
    import sys
    code = r'''
import ctypes as C, sys
sys.path.insert(0, %r)
import mpi_pastar_msa_b200 as m
from mpi_pastar_msa_b200 import api
L = C.CDLL(m.lib_path())
z = C.c_void_p(0)
getters = {"pg_search_outbox_capacity", "pg_search_region_bytes", "pg_xrec_stride", "pg_ctx_destroy", "pg_allow_extended_n"}
skip = {"pg_release_cached_memory", "pg_default_cost_table", "pg_abi_version", "pg_last_error"}
for name in sorted(api.EXPORTS):
    if name in skip:
        continue
    f = getattr(L, name)
    f.restype = C.c_int64 if name in ("pg_search_outbox_capacity", "pg_search_region_bytes") else C.c_int
    r = f(z, z, z, z, z, z, z, z, z, z)
    assert r == (0 if name in getters else 1), (name, r)
L.pg_last_error.restype = C.c_char_p
assert isinstance(L.pg_last_error(z), bytes)
print("ok")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300)
    assert r.returncode == 0 and r.stdout.decode().strip() == "ok", (r.returncode, r.stderr.decode()[-1500:])


def test_ctx_create_validates_the_problem_before_touching_the_device():
    """N outside {3..10, 14, 16} (msa_pastar_main.cpp:34-36; 11, 12, 13, 15 need pg_allow_extended_n) and empty sequences are
    PG_ERR_ARG on any box - also where there is no device, i.e. the check does not depend on CUDA."""
    for seqs in (["AC", "AD"], ["AC"] * 17, ["AC"] * 11, ["AC", "AD", ""]):
        with pytest.raises(api.PastarError) as e:
            m.PastarGPU(seqs, weights=None)
        assert "PG_ERR_ARG" in str(e.value)
