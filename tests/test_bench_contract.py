"""bench.py's reference arm runs on host cores only (no GPU): its JSON line keeps the driver's contract.

The GPU arm's line is produced on the GPU box (profiles/r02_bench_n*.json); here only the CPU leg can run.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_ref():
    sys.path.insert(0, ROOT)
    from oracle import refio
    return refio.available()


def _run(env_extra=None):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    env.update(env_extra or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    return r


@pytest.mark.skipif(not _have_ref(), reason="oracle/_ref is built by __graft_entry__.build() where /root/reference exists")
def test_reference_arm_line():
    r = _run()
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    lines = [ln for ln in r.stdout.decode().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "node_expansions_per_sec" and d["unit"] == "expansions/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == d["value"] and cb["sample"]
    # SURVEY 8(d) micro-baselines, one core, reference code only
    mb = cb["micro"]
    assert mb["cores"] == 1 and mb["pair_align_gcups"] > 0 and mb["getneigh_parents_per_s"] > 0
    assert "S7" in d["config"]["workload"] or "N=7" in d["config"]["workload"]
    assert set(d["reference_build"]) >= {"mpicxx", "mpiexec", "boost_headers", "lz4_header", "buildable"}


def test_steps_below_one_are_refused():
    for args in (["--steps", "0"], ["--steps", "-3", "--impl", "reference"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, timeout=120)
        assert r.returncode == 2 and b"--steps must be at least 1" in r.stderr, r.stderr.decode()[-2000:]


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    """--dump-outputs writes the timed rounds' results after exactly --steps timed rounds, on the same inputs every run."""
    runs = []
    for k in (1, 2):
        d = tmp_path / ("run%d" % k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "3", "--quick",
                            "--batch", "4096", "--table-capacity", str(1 << 24), "--dump-outputs", str(d)],
                           cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        line = json.loads([ln for ln in r.stdout.decode().splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 5
        out = {p.stem: np.load(p) for p in d.glob("*.npy")}
        assert set(out) == {"search_status", "node_pos", "node_g", "node_parenti"}
        assert all(a.dtype == np.float64 for a in out.values()) and sum(a.nbytes for a in out.values()) <= 64 << 20
        # status = [min open f, best goal g, finished, g, f, pops, expansions, ..., rounds, ...]: ramp-up + warm-up + timed
        assert out["search_status"][11] == line["config"]["ramp_up_rounds_untimed"] + 3 + 5
        found = out["node_g"] >= 0
        assert found.any() and (out["node_g"][found] > 0).all()
        assert ((out["node_parenti"][found] >= 1) & (out["node_parenti"][found] < 128)).all()
        runs.append(out)
    assert np.array_equal(runs[0]["node_pos"], runs[1]["node_pos"])
    # what the device computed and bench.search_outputs documents as exact from run to run: the min open f, and the
    # values of the sampled nodes that are settled (g + h below the min open f: closed with their final g)
    min_f = runs[0]["search_status"][0]
    assert runs[1]["search_status"][0] == min_f
    from conftest import S7
    from oracle import oracle as O
    P = O.Problem(S7())
    h = np.array([P.calculate_h(p) for p in runs[0]["node_pos"].astype(np.uint16)])
    settled = [(r["node_g"] >= 0) & (r["node_g"] + h < min_f) for r in runs]
    assert np.array_equal(settled[0], settled[1]) and settled[0].any()
    for name in ("node_g", "node_parenti"):
        assert np.array_equal(runs[0][name][settled[0]], runs[1][name][settled[0]]), name


@pytest.mark.skipif(not _have_ref(), reason="oracle/_ref is built by __graft_entry__.build() where /root/reference exists")
def test_reference_arm_other_ranks_do_no_work():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29571"})
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert not [ln for ln in r.stdout.decode().splitlines() if ln.startswith("{")]
