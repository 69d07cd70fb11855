"""CPU: the host mirror's FASTA reader and result printer against the reference's own read_fasta.cpp / backtrace.cpp.

`mpi_pastar_msa_b200/bin/host_cpu_test` (tests/cpp/host_cpu_test.cpp + the CLI's translation unit) and `oracle/_ref/pastar_ref`
(unmodified reference sources) are given the same files; their stdout must be byte-identical - through a pipe (one unwrapped
block, backtrace.cpp:26-27) and on pseudo-terminals of several widths (blocks of columns - 1, backtrace.cpp:30-31).
Without that build the reference's output is known by its digest (tests/golden/ref_comparisons.json.gz, tests/refdata.py).
"""
import fcntl
import os
import pty
import random
import struct
import subprocess
import termios

import pytest

from conftest import ROOT
import refdata as D

OURS = os.path.join(ROOT, "mpi_pastar_msa_b200", "bin", "host_cpu_test")
REF = os.path.join(ROOT, "oracle", "_ref", "pastar_ref")


def _pipe(argv):
    r = subprocess.run(argv, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120)
    return r.returncode, r.stdout


def _on_tty(argv, cols):
    """Run with stdin and stdout on a pseudo-terminal `cols` wide; return what it wrote (CR LF -> LF)."""
    master, slave = pty.openpty()
    fcntl.ioctl(slave, termios.TIOCSWINSZ, struct.pack("HHHH", 24, cols, 0, 0))
    p = subprocess.Popen(argv, stdin=slave, stdout=slave, stderr=subprocess.PIPE, close_fds=True)
    os.close(slave)
    out = b""
    while True:
        try:
            chunk = os.read(master, 65536)
        except OSError:
            break
        if not chunk:
            break
        out += chunk
    p.wait(timeout=120)
    os.close(master)
    return p.returncode, out.replace(b"\r\n", b"\n")


def _rows(n, cols, seed, dash=0.2):
    rng = random.Random(seed)
    base = [rng.choice("ACDEFGHIKLMNPQRSTVWY") for _ in range(cols)]
    rows = []
    for _ in range(n):
        rows.append("".join("-" if rng.random() < dash else (c if rng.random() < 0.7 else rng.choice("ACDEFGHIKLMNPQRSTVWY")) for c in base))
    return rows


def _fasta_for(n, path):
    with open(path, "w") as f:
        for i in range(n):
            f.write(">s%d\nACD\n" % i)


def test_check_program_is_built():
    assert os.path.exists(OURS), "python -m mpi_pastar_msa_b200.build"


def _same_as_reference(what, args, ref_argv, got, run=_pipe, *run_args):
    """got = (rc, stdout) of our program; the reference's comes from running ref_argv, or from the stored digest."""
    want = D.program_output(what, args, lambda: run(ref_argv, *run_args), lambda: got)
    return want == [0, D.digest(got[1])] and got[0] == 0


@pytest.mark.parametrize("n,cols,seed", [(3, 1, 1), (3, 59, 2), (5, 300, 3), (8, 12, 4), (10, 79, 5), (14, 80, 6), (16, 161, 7), (4, 2000, 8)])
def test_similarity_and_alignment_print(tmp_path, n, cols, seed):
    rows = _rows(n, cols, seed)
    rp, fa = str(tmp_path / "rows.txt"), str(tmp_path / "n.fasta")
    open(rp, "w").write("\n".join(rows) + "\n")
    _fasta_for(n, fa)  # the reference's printer is a template in N: the FASTA file only selects the instantiation
    got = _pipe([OURS, "print", rp])
    assert _same_as_reference("print", (n, cols, seed, "pipe"), [REF, "print", fa, rp], got)
    lines = got[1].decode().split("\n")
    assert lines[0].startswith("Similarity: ") and lines[1] == "" and lines[2:2 + n] == rows  # not a tty: one block
    for width in (20, 41, 80, 81, 200):
        got = _on_tty([OURS, "print", rp], width)
        assert _same_as_reference("print", (n, cols, seed, width), [REF, "print", fa, rp], got, _on_tty, width), width
        blocks = -(-cols // (width - 1))
        assert got[1].count(b"\n") == 1 + blocks * (n + 1)


def test_similarity_extremes(tmp_path):
    fa = str(tmp_path / "n.fasta")
    _fasta_for(3, fa)
    for rows in (["AAAA", "AAAA", "AAAA"], ["ACDE", "CDEA", "DEAC"], ["A---", "-C--", "--D-"], ["----", "----", "AAAA"]):
        rp = str(tmp_path / "rows.txt")
        open(rp, "w").write("\n".join(rows) + "\n")
        assert _same_as_reference("print", (3, rows), [REF, "print", fa, rp], _pipe([OURS, "print", rp]))


FASTA_FILES = {
    "plain": ">a\nACD\n>b\nACE\n>c\nAC\n",
    "multi_line_records": ">a desc\nACD\nEFG\n>b\nAC\nE\n>c\nA\n",
    "no_trailing_newline": ">a\nACD\n>b\nACE\n>c\nAC",
    "blank_lines_split_records": ">a\nAC\n\nGT\n>b\nTT\n\n\n>c\nGG\n",   # read_fasta.cpp:20-24: an empty line ends a record too
    "empty_records_dropped": ">a\n>b\nAC\n>c\n>d\nGG\n>e\nTT\n",
    "no_header_first": "ACD\n>b\nACE\n>c\nAC\n",
    "header_only_tail": ">a\nACD\n>b\nACE\n>c\nAC\n>d\n",
    "sixteen": "".join(">s%d\n%s\n" % (i, "ACDEFGHIKL"[: 1 + i % 7]) for i in range(16)),
}


@pytest.mark.parametrize("name", list(FASTA_FILES))
def test_read_fasta_file_matches_reference(tmp_path, name):
    fa = str(tmp_path / "in.fasta")
    open(fa, "w").write(FASTA_FILES[name])
    got = _pipe([OURS, "seqs", fa])
    assert _same_as_reference("seqs", (FASTA_FILES[name],), [REF, "seqs", fa], got), got
    # and the Python reader used by tests / bench agrees with both
    import mpi_pastar_msa_b200 as m
    seqs = m.read_fasta(fa)
    assert got[1].decode().split("\n")[:-1] == [str(len(seqs))] + seqs
