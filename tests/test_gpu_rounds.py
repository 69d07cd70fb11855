"""Round accounting and the CUDA-graph replay of round groups: pg_search_rounds, pg_search and pg_multi_search replay
captured groups of rounds unless PG_NO_GRAPH is set, and a graph must change neither the rounds counted nor the result."""
import numpy as np
import pytest

from conftest import CASES, KNOWN_OPT, weighted_sp_score

pytestmark = pytest.mark.gpu

CAP = {"PF08184": 1 << 22, "kinase": 1 << 27}


def _graphs(monkeypatch, on):
    if on:
        monkeypatch.delenv("PG_NO_GRAPH", raising=False)
    else:
        monkeypatch.setenv("PG_NO_GRAPH", "1")


@pytest.mark.parametrize("graph", [True, False])
def test_search_rounds_counts_every_round(gpu_lib, monkeypatch, graph):
    """20 rounds are 2 replays of a group of 8 and 4 plain rounds with graphs, 20 plain rounds without; a new f_limit
    captures a new group."""
    _graphs(monkeypatch, graph)
    with gpu_lib.PastarGPU(CASES["kinase"]) as G:
        G.build_pair_tables()
        G.search_begin(table_capacity=1 << 22, batch_target=64)
        G.search_rounds(20)
        assert G.search_status()[2]["rounds"] == 20
        G.search_rounds(20, f_limit=2**31 - 2)
        assert G.search_status()[2]["rounds"] == 40
        G.search_rounds(20)
        assert G.search_status()[2]["rounds"] == 60
        G.search_end()


@pytest.mark.parametrize("name", ["PF08184", "kinase"])
def test_search_same_with_and_without_graphs(gpu_lib, monkeypatch, name):
    seqs = CASES[name]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        out = []
        for graph in (True, False):
            _graphs(monkeypatch, graph)
            out.append(G.search(table_capacity=CAP[name], batch_target=16384))
        for r in out:
            assert r["finished"] == 1 and r["g"] == r["lower_bound"] == KNOWN_OPT[name]
            assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"]


def test_search_batch_one_repeats_with_and_without_graphs(gpu_lib, monkeypatch):
    """One parent per round: the search is the same sequence of expansions whichever way its rounds are launched."""
    seqs = CASES["PF08184"]
    with gpu_lib.PastarGPU(seqs) as G:
        G.build_pair_tables()
        out = []
        for graph in (True, True, False):
            _graphs(monkeypatch, graph)
            out.append(G.search(table_capacity=1 << 22, batch_target=1))
        for r in out:
            assert r["finished"] == 1 and r["g"] == r["lower_bound"] == KNOWN_OPT["PF08184"]
            assert weighted_sp_score(seqs, G.w_int, r["rows"]) == r["g"]
            assert (r["expansions"], r["rounds"]) == (out[0]["expansions"], out[0]["rounds"])


@pytest.mark.parametrize("name,batch", [("PF08184", 64), ("kinase", 16384)])
def test_multi_search_same_with_and_without_graphs(gpu_lib, monkeypatch, name, batch):
    seqs = CASES[name]
    Gs = []
    for _ in range(2):
        G = gpu_lib.PastarGPU(seqs)
        G.build_pair_tables()
        G.configure_hash("FZORDER", 12)
        Gs.append(G)
    w = gpu_lib.host_weights(seqs).astype(np.int32)
    for graph in (True, False):
        _graphs(monkeypatch, graph)
        tot, per = gpu_lib.multi_search(Gs, table_capacity=1 << 25, batch_target=batch)
        assert tot["finished"] == 1 and tot["g"] == tot["lower_bound"] == KNOWN_OPT[name]
        assert weighted_sp_score(seqs, w, tot["rows"]) == tot["g"]
        assert sum(p["expansions"] for p in per) == tot["expansions"]
    for G in Gs:
        G.close()
