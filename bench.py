#!/usr/bin/env python
"""bench.py — node expansions/s of the batched PA-Star search on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[3], synthetic N=7 x length 500 random protein (seed 12345),
PAM250 costs, Altschul weights, budgeted A* search (random sets never terminate: SURVEY §7).
A step = one search round of the hot path: pop `batch` frontier nodes -> expand all 2^N-1 successors of each
(g via weighted SP, h via pairwise tables, owner) -> closed/open-table dedupe -> push survivors (+ exchange for N>1).
value  = expansions in the K timed steps / device time (state resident in HBM), whole job over all ranks.
e2e    = same metric through the C ABI from HOST buffers: context create (H2D of sequences, cost, weights), pairwise
         tables, table set-up (buffers from the library cache, cleared), search from the start node to an expansion budget, result D2H; wall clock around the
         calls (N > 1: the same through mpi_pastar_msa_b200.dist, per-rank set-up included).
roofline = the round's dominant kernel (expand + probe) against the measured HBM copy bandwidth (MEASURED_PEAKS.json);
         roofline.kernels lists select / claim / expand+probe / insert with their CUDA-event times and algorithmic bytes.
cpu_baseline / --impl reference = the reference's own getNeigh / PairAlign / weights (oracle/_ref, compiled from
         the unmodified sources) under the restated T-thread hash-partitioned driver, on this box's host cores.
--dump-outputs DIR (N = 1) = after the K timed rounds, what they leave a caller of the search (see search_outputs) as
         DIR/<name>.npy in float64, so that two builds can be compared output for output on identical inputs.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG", "WARN")  # default only: the driver may ask for INFO to check the ranks
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's own lines go to stderr: stdout carries the one JSON line

import numpy as np  # noqa: E402

AA = "ACDEFGHIKLMNPQRSTVWY"
METRIC, UNIT = "node_expansions_per_sec", "expansions/s"
N_SEQ, LENGTH, SEED = 7, 500, 12345
WORKLOAD = "synthetic N=7 x L=500 random protein (seed 12345), PAM250 costs, Altschul weights, budgeted A* search"
CPU_STEP_POPS = 15000  # the reference arm's step: a bounded sample of the same search (100 steps = 1.5 M dequeues: ~15 s on the 16 host threads of the GPU box)


def s7_seqs():
    import random
    r = random.Random(SEED)
    return ["".join(r.choice(AA) for _ in range(LENGTH)) for _ in range(N_SEQ)]


STATUS_FIELDS = ("finished", "g", "f", "pops", "expansions", "generated", "reopen", "open_size", "closed_size", "rounds",
                 "probed", "pushed", "inserted", "survivors")  # pg_result counters; the timing fields are left out
DUMP_NODES, DUMP_DEPTH = 4096, 4


def search_outputs(G):
    """What the search rounds so far give their caller: pg_search_status (min open f, best goal g, counters) and, through
    pg_search_lookup, the g and parenti (-1 when absent) of DUMP_NODES lattice nodes within DUMP_DEPTH moves of the
    start, drawn with a fixed seed.  The min open f and the values of settled nodes (g + h below the min open f: closed
    with their final g; all of the sample in the default configuration) repeat exactly from run to run; pops, expansions
    and the other counters vary in about the fifth digit, because concurrent inserts of one node race to the table."""
    min_f, goal, c = G.search_status()
    rng = np.random.default_rng(SEED)
    moves = rng.integers(1, 1 << G.n, (DUMP_NODES, DUMP_DEPTH))
    moves[np.arange(DUMP_DEPTH) >= rng.integers(1, DUMP_DEPTH + 1, (DUMP_NODES, 1))] = 0
    pos = ((moves[:, :, None] >> np.arange(G.n)) & 1).sum(axis=1).astype(np.uint16)
    vals = np.array([G.search_lookup(p) or (-1, -1) for p in pos], dtype=np.float64).reshape(DUMP_NODES, 2)
    return {"search_status": np.array([min_f, goal] + [c[k] for k in STATUS_FIELDS], dtype=np.float64),
            "node_pos": pos.astype(np.float64), "node_g": vals[:, 0], "node_parenti": vals[:, 1]}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons DURING the timed region (NVML, ~5 ms period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        for k, bit in names.items():
            if r & bit:
                self.reasons.add(k)

    def run(self):
        if not self.nv:
            return
        while not self.stop_flag:
            try:
                self.sample()
            except Exception:
                break
            time.sleep(0.005)

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_reference_run(threads, steps, warmup, want_sample=True):
    """The reference CPU path on S7: oracle/_ref (reference arithmetic + restated T-thread driver), else the C port."""
    from oracle import refio
    seqs = s7_seqs()
    budget = (steps + warmup) * CPU_STEP_POPS
    if refio.available():
        r = refio.pastar(seqs, threads, budget, "FZORDER", 12, timeout=1800, warm_pops=max(1, warmup * CPU_STEP_POPS))
        secs, exps = r["timed_seconds"], r["timed_expansions"]
        kind, cores = "reference", threads
        what = ("oracle/_ref: reference Node::getNeigh/PairAlign/weights under the restated hash-partitioned PA-Star driver "
                "(PAStar.cpp:319-547; Boost/MPI absent), %d threads x 1 rank" % threads)
    else:
        from oracle import oracle as O
        P = O.Problem(seqs)
        P.astar(budget=max(1, warmup * CPU_STEP_POPS), want_rows=False)
        t0 = time.time()
        r = P.astar(budget=budget, want_rows=False)
        secs, exps = time.time() - t0, r["expansions"]
        kind, cores = "port", 1
        what = "oracle/pastar_oracle.c serial A* (AStar.cpp:53-104 restated), 1 thread"
    return {"value": exps / secs if secs > 0 else 0.0, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%s; %d dequeues timed after %d warm-up dequeues of the S7 search" % (what, steps * CPU_STEP_POPS, warmup * CPU_STEP_POPS),
            "seconds": secs, "expansions": exps}


def cpu_micro_baselines(seconds=2.0):
    """SURVEY 8(d) micro-baselines on ONE host core, reference code only (oracle/_ref `micro`): PairAlign::Align GCUPS over the
    21 S7 tables and Node::getNeigh parents/s on 4096 seeded interior parents.  Reported beside cpu_baseline, never a target."""
    from oracle import refio
    if not refio.available():
        return {"unavailable": "oracle/_ref not built"}
    r = refio.micro(s7_seqs(), seconds)
    return {"cores": 1, "pair_align_gcups": r["dp_gcups"], "pair_align_seconds_s7": r["dp_seconds"],
            "getneigh_parents_per_s": r["neigh_parents_per_s"],
            "getneigh_successors_per_s": r["neigh_successors"] / r["neigh_seconds"] if r["neigh_seconds"] > 0 else None,
            "sample": "reference PairAlign::Align over the 21 S7 tables (%d cells) and Node<7>::getNeigh over 4096 seeded interior "
                      "parents, ~%.0f s each on one core" % (r["dp_cells"], seconds / 2)}


def probe_reference_toolchain():
    """BASELINE.md 4 step 1: can the real reference (mpich + Boost + LZ4, `make` -> ./bin/pastar) be built on this box?  Its
    sources are not on the GPU box (/root/reference exists only in the build container), so even a complete toolchain could
    only build it there; recorded so that the baseline's kind is never a guess."""
    import shutil
    have = {"mpicxx": bool(shutil.which("mpicxx") or shutil.which("mpic++")), "mpiexec": bool(shutil.which("mpiexec")),
            "boost_headers": any(os.path.exists(os.path.join(d, "boost", "multi_index_container.hpp")) for d in ("/usr/include", "/usr/local/include")),
            "lz4_header": any(os.path.exists(os.path.join(d, "lz4.h")) for d in ("/usr/include", "/usr/local/include")),
            "reference_sources": os.path.exists("/root/reference/pastar/PAStar.cpp")}
    have["buildable"] = all(have.values())
    return have


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    steps = args.steps
    t0 = time.time()
    b = cpu_reference_run(threads, steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": b["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * b["seconds"] / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "step": "%d dequeues of the CPU search" % CPU_STEP_POPS, "threads": threads, "ranks": 1,
                       "nproc": os.cpu_count()},
            "cpu_baseline": {k: b[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": b["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.time() - t0, "reference_build": probe_reference_toolchain()}
    try:
        line["cpu_baseline"]["micro"] = cpu_micro_baselines()
    except Exception as ex:
        line["cpu_baseline"]["micro"] = {"error": repr(ex)}
    print(json.dumps(line), flush=True)


# Known answers of the reference's own fixtures (SURVEY.md 4: reference arithmetic, optimal g*), used by the N > 1 parity gate.
PARITY_INPUTS = {
    "PF08184": (["QAVRYANGYTYDIETGQVSSPYTGRVYETKGKAPFYGFGFEHPYHYYPGYYHGYPHAFY",
                 "QAVRYADGYTYDIETGQVSSPYTGRVYETKGKAPFYGFGFEHPYHYYPGYYHGYPHAFY",
                 "QAVRYANGYTYDIETGQVSSPYTGRVYETKGKAPFYGFGFKYPYHYYPGYYHGYPHVFY"], 24450, 1 << 22, 64),
    "kinase": ([
        "NYIFGRTLGAGSFGVVRQARKLSTNEDVAIKILLKKALQGNNVQLQMLYEELSILQKLSHPNIVSFKDWFESKDKFYIVTQLATGGELFDRILSRGKFTEVDAVEIIVQILGAVEYMHSKNVVHRDLKPENVLYVDKSENSPLVIADFGIAKQLKGEEDLIYKAAGSLGYVAPEVLTQDGHGKPCDIWSIGVITYTLLCGYSPFIAESVEGFMEECTASRYPVTFHMPYWDNISIDVKRFILKALRLNPADRPTATELLDDPWITSK",
        "DFEILKVIGRGAFSEVAVVKMKQTGQVYAMKIMNKWDMLKRGEVSCFREERDVLVNGDRRWITQLHFAFQDENYLYLVMEYYVGGDLLTLLSKFGERIPAEMARFYLAEIVMAIDSVHRLGYVHRDIKPDNILLDRCGHIRLADFGSCLKLRADGTVRSLVAVGTPDYLSPEILQAVGGGPGTGSYGPECDWWALGVFAYEMFYGQTPFYADSTAETYGKIVHYKEHLSLPLVDEGVPEEARDFIQRLLCPPETRLGRGGAGDFRTHPFFFGLDWD",
        "TRKFKVELGRGESGTVYKGVLEDDRHVAVKKLENVRQGKEVFQAELSVIGRINHMNLVRIWGFCSEGSHRLLVSEYVENGSLANILFSEGGNILLDWEGRFNIALGVAKGLAYLHHECLEWVIHCDVKPENILLDQAFEPKITDFGLVKLLNRGGSTQNVSHVRGTLGYIAPEWVSSLPITAKVDVYSYGVVLLELLTGTRVSELVGGTDEVHSMLRKLVRMLSAKLEGEEQSWIDGYLDSKLNRPVNYVQARTLIKLAVSCL",
        "QIRLTGRVGSGRFGNVSRGDYRGEAVAVKVFNALDEPAFHKETEIFETRMLRHPNVLRYIGSDRVDTGFVTELWLVTEYHPSGSLHDFLLENTVNIETYYNLMRSTASGLAFLHNQIGGSKESNKPAMAHRDIKSKNIMVKNDLTCAIGDLGLSLSKPEDAASDIIANENYKCGTVRYLAPEILNSTMQFTVFESYQCADVYSFSLVMWETLCRCEDGDVLPREAATVIPYIEWTDRDPQDAQMFDVVCTRRLRPTENPLWKDHPEMKHIMEI",
        "HYKVGRRIGEGSFGVIFEGTNLLNNQQVAIKFEPRRSDAPQLRDEYRTYKLLAGCTGIPNVYYFGQEGLHNVLVIDLLGPSLEDLLDLCGRKFSVKTVAMAAKQMLARVQSIHEKSLVYRDIKPDNFLIGRPNSKNANMIYVVDFGMVKFYRDPVTKQHIPYREKKNLSGTARYMSINTHLGREQSRRDDLEALGHVFMYFLRGSLPWQGLKAATNKQKYERIGEKKQSTPLRELCAGFPEEFYKYMHYARNLAFDATPDYDYLQGLFSKVL"],
        421546, 1 << 26, 16384),
}


def multi_gpu_parity(m, dist, world, rank, local):
    """N > 1 parity on the real devices, before anything is timed: PF08184.fasta (BASELINE configs[2]) and kinase.fasta
    solved to the optimality-preserving stop through PartitionedSearch.run() in all three exchange modes - NCCL
    all-to-all of successor records (what replaces PAStarSender.cpp:62 / PAStarReceiver.cpp:55), P2P successor records,
    P2P parent forwarding - each checked against the reference's optimal cost and by re-scoring the alignment."""
    import torch
    from mpi_pastar_msa_b200.dist import CudaEngine, CudaEngineP2P, PartitionedSearch
    out, ok = {}, True
    for name, (seqs, g_ref, cap, batch) in PARITY_INPUTS.items():
        G = m.PastarGPU(seqs, device=local)
        G.build_pair_tables()
        G.configure_hash("FZORDER", 12)  # the reference's defaults (CoordHash.cpp:17-18)
        per = {}
        for mode in ("nccl_all_to_all", "p2p_records", "p2p_parent_forwarding"):
            try:
                if mode == "nccl_all_to_all":
                    eng = CudaEngine(G, world, rank, cap, batch)
                else:
                    eng = CudaEngineP2P(G, world, rank, dist, cap, batch, forward=mode == "p2p_parent_forwarding")
                drv = PartitionedSearch(eng, dist, seqs, lambda pos: int(G.owner(np.array(pos, dtype=np.uint16), world)[0]))
                r = drv.run()
                eng.end()
                good = r["finished"] == 1 and r["g"] == g_ref and m.rescore_alignment(seqs, G.w_int, r["rows"]) == g_ref
                per[mode] = {"ok": bool(good), "g": r["g"], "expansions": r["expansions"], "rounds": r["rounds"]}
            except Exception as ex:  # a mode that cannot run is a failure, not a skip
                per[mode] = {"ok": False, "error": repr(ex)}
            t = torch.tensor([1 if per[mode]["ok"] else 0], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)  # every rank must agree
            per[mode]["ok"] = bool(t.item())
            ok = ok and per[mode]["ok"]
        per["g_reference"] = g_ref
        out[name] = per
        G.close()
    out["status"] = "ok" if ok else "FAILED"
    out["n_gpus"] = world
    return out


def run_ours(args, rank, world):
    import torch
    import mpi_pastar_msa_b200 as m
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    parity = None
    if world > 1 and not args.skip_parity:
        parity = multi_gpu_parity(m, dist, world, rank, local)
        if parity["status"] != "ok":
            if rank == 0:
                print(json.dumps({"metric": METRIC, "value": None, "n_gpus": world, "parity": parity, "error": "multi-GPU parity failed"}), flush=True)
            dist.barrier()
            dist.destroy_process_group()
            raise SystemExit(3)

    seqs = s7_seqs()
    batch, cap = args.batch, args.table_capacity
    K, W = args.steps, max(3, args.warmup)
    stream = torch.cuda.current_stream()

    G = m.PastarGPU(seqs, device=local)
    G.set_stream(stream.cuda_stream)
    dp_ms = min(G.build_pair_tables() for _ in range(3))
    cells = sum((len(a) + 1) * (len(b) + 1) for i, a in enumerate(seqs) for b in seqs[i + 1:])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    launches_per_step = 4  # select + claim + expand/probe + insert
    extra = {}
    if world == 1:
        G.search_begin(1, 0, cap, batch)
        # ---- ramp-up (untimed): grow the frontier from the start node until rounds pop full batches
        ramp = 0
        while True:
            before = G.search_status()[2]["pops"]
            G.search_rounds(8)
            ramp += 8
            if G.search_status()[2]["pops"] - before >= 8 * batch or ramp > 4000:
                break
        G.search_rounds(W)
        # ---- pass 1, the timed region of `value`: K rounds as the product runs them (groups of 8 rounds replayed as a CUDA
        # graph, as in pg_search), CUDA events on the launching stream around them
        v0 = G.search_status()[2]
        sampler = ClockSampler(local)
        sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        G.search_rounds(K)
        e1.record(stream)
        barrier()
        sampler.stop_flag = True
        max_ms = e0.elapsed_time(e1)
        v1 = G.search_status()[2]
        total_exp = v1["expansions"] - v0["expansions"]
        dv = {k: v1[k] - v0[k] for k in ("expansions", "generated", "probed", "pushed", "pops")}
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in search_outputs(G).items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        # ---- pass 2, the per-kernel times behind `roofline`: the next K rounds with an event pair around every launch
        # (plain launches: the extra events would sit between graph nodes)
        c0 = G.search_status()[2]
        G.search_profile(True)
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        G.search_rounds(K)
        p1.record(stream)
        barrier()
        ms = p0.elapsed_time(p1)
        c1 = G.search_status()[2]
        G.search_profile(False)
        d = {k: c1[k] - c0[k] for k in ("expansions", "generated", "probed", "pushed", "pops")}
        expand_ms, select_ms = c1["expand_ms"] - c0["expand_ms"], c1["select_ms"] - c0["select_ms"]
        claim_ms, insert_ms = c1["claim_ms"] - c0["claim_ms"], c1["insert_ms"] - c0["insert_ms"]
        extra["profiled_pass"] = {"ms_per_step": ms / K, "expansions_per_sec": d["expansions"] / (ms * 1e-3),
                                  "note": "the K rounds after the timed ones, with per-launch events (no graph): the source of roofline.kernels"}
        G.search_end()
    else:
        from mpi_pastar_msa_b200.dist import CudaEngine, CudaEngineP2P, PartitionedSearch
        fwd = os.environ.get("PG_FWD", "1") == "1"

        def make_engine(gpu, hash_type, hash_shift):
            gpu.configure_hash(hash_type, hash_shift)
            try:  # fused expansion + exchange over peer-mapped inboxes; NCCL all-to-all if symmetric memory is unavailable
                if os.environ.get("PG_P2P", "1") == "0":
                    raise RuntimeError("PG_P2P=0")
                e = CudaEngineP2P(gpu, world, rank, dist, cap, batch, forward=fwd)
                how = ("device-driven parent forwarding: the claim kernel stores each live parent into the peer-mapped inbox (NVLink) of "
                       "every partition owning one of its successors; counts published by a device kernel, one symmetric-memory barrier per round"
                       if fwd else
                       "device-driven: p2p stores of successor records into peer-mapped inboxes (NVLink) from the expand kernel, counts "
                       "published by a device kernel, one symmetric-memory barrier per round")
            except Exception as ex:
                e = CudaEngine(gpu, world, rank, cap, batch)
                how = "nccl all_to_all_single (p2p unavailable: %r)" % (ex,)
            return e, how

        def timed_partitioned(gpu, hash_type, hash_shift, k_steps, w_steps, sample_clocks):
            """Ramp the partitioned search up from the start node (untimed), then time k_steps rounds on the device."""
            e, how = make_engine(gpu, hash_type, hash_shift)
            dr = PartitionedSearch(e, dist, seqs, lambda pos: int(gpu.owner(np.array(pos, dtype=np.uint16), world)[0]))
            ch = getattr(e, "async_rounds", False)  # device-driven rounds: one status exchange per call, not per round
            rmp = 0
            while True:
                _, _, t0_ = dr.step(rounds=8 if ch else 1)
                _, _, t1_ = dr.step(rounds=8 if ch else 1)
                rmp += 16 if ch else 2
                if t1_[2] - t0_[2] >= (8 if ch else 1) * world * batch or rmp > 4000:
                    break
            dr.step(rounds=w_steps)
            _, _, t0_ = dr.step()
            # pass 1, the timed region of `value`: k_steps rounds as the product runs them (device-driven; groups of 8 rounds
            # replayed as a CUDA graph, dist.CudaEngineP2P.rounds), one status exchange at the end
            smp = ClockSampler(local) if sample_clocks else None
            if smp:
                smp.start()
            barrier()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0 = dr.bytes_sent
            ev0.record(stream)
            if ch:
                _, _, t1_ = dr.step(rounds=k_steps)
            else:
                for _ in range(k_steps):
                    _, _, t1_ = dr.step()
            ev1.record(stream)
            barrier()
            if smp:
                smp.stop_flag = True
            tt = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sent1 = dr.bytes_sent
            # pass 2, rank 0's per-kernel times: the next k_steps rounds with an event pair around every launch (plain launches)
            gpu.search_profile(True)
            p0 = gpu.search_status()[2]
            if ch:
                dr.step(rounds=k_steps)
            else:
                for _ in range(k_steps):
                    dr.step()
            p1 = gpu.search_status()[2]
            gpu.search_profile(False)
            out = {"max_ms": float(tt.item()), "tot0": t0_, "tot1": t1_, "ramp": rmp, "how": how, "sampler": smp,
                   "nvlink_bytes_per_step_per_gpu": (sent1 - s0) / k_steps,
                   "rank0_kernel_ms_per_step": {k: (p1[k] - p0[k]) / k_steps for k in ("select_ms", "claim_ms", "expand_ms", "insert_ms", "inbox_ms")},
                   "rank0_records_inserted_per_step": (p1["survivors"] - p0["survivors"]) / k_steps,
                   "rank0_counts_per_step": {k: (p1[k] - p0[k]) / k_steps for k in ("pops", "expansions", "probed", "pushed", "survivors")},
                   "forward": isinstance(e, CudaEngineP2P) and e.forward, "p2p": isinstance(e, CudaEngineP2P)}
            e.end()
            return out

        r_main = timed_partitioned(G, args.hash_type, args.hash_shift, K, W, True)
        extra["exchange"] = r_main["how"]
        if r_main["forward"]:
            launches_per_step = 7  # select, claim, forward, publish counts, expand (own), expand (forwarded), insert
        elif r_main["p2p"]:
            launches_per_step = 5 + (world - 1)  # select, claim, expand/probe, insert (local), publish counts + one insert per source
        else:
            launches_per_step = 6  # select, claim, expand/probe, insert (local), insert (received), status select
        ramp, sampler, max_ms = r_main["ramp"], r_main["sampler"], r_main["max_ms"]
        tot0, tot1 = r_main["tot0"], r_main["tot1"]
        total_exp = tot1[0] - tot0[0]
        d = {"expansions": total_exp, "generated": tot1[1] - tot0[1], "pops": tot1[2] - tot0[2]}
        for k in ("nvlink_bytes_per_step_per_gpu", "rank0_kernel_ms_per_step", "rank0_records_inserted_per_step"):
            extra[k] = r_main[k]
        expand_ms = select_ms = None
        # the same measurement under the reference's default owner hash (FZORDER shift 12, CoordHash.cpp:17-18) and the
        # round-1 setting (FZORDER shift 17), shorter: the owner hash decides how many parents straddle partitions
        if not args.no_hash_sweep:
            sweep = {}
            for ht, sh in (("FZORDER", 12), ("FZORDER", 17)):
                if (ht, sh) == (args.hash_type, args.hash_shift):
                    continue
                try:
                    rs = timed_partitioned(G, ht, sh, max(5, K // 4), W, False)
                    ex_ = rs["tot1"][0] - rs["tot0"][0]
                    sweep["%s shift %d" % (ht, sh)] = {"value": ex_ / (rs["max_ms"] * 1e-3), "unit": UNIT, "ms_per_step": rs["max_ms"] / max(5, K // 4),
                                                       "steps": max(5, K // 4), "nvlink_bytes_per_step_per_gpu": rs["nvlink_bytes_per_step_per_gpu"],
                                                       "rank0_kernel_ms_per_step": rs["rank0_kernel_ms_per_step"]}
                except Exception as ex:
                    sweep["%s shift %d" % (ht, sh)] = {"error": repr(ex)}
            extra["owner_hash_sweep"] = sweep

    value = total_exp / (max_ms * 1e-3)
    clocks = sampler.result()
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": max_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": batch, "table_slots_per_gpu": cap, "parallelism": "hash-partition x%d" % world + ("" if world == 1 else " (%s shift %d)" % (args.hash_type, args.hash_shift)),
                       "ramp_up_rounds_untimed": ramp,
                       "l2": "inputs larger than L2: %.1f GiB of value blocks per GPU (4 four-byte slots per coordinate), ~1 GB of distinct 128-byte lines touched per step"
                             % (cap * 16 / 2**30)},
            "clocks": clocks, "gpu_launches": launches_per_step * K,
            "successors_per_sec": (dv if world == 1 else d)["generated"] / (max_ms * 1e-3)}

    if world > 1:
        # roofline of the round on rank 0 (the per-launch split of the two expand launches is not timed separately at N > 1):
        # the algorithmic bytes of DESIGN.md 4 for claim + both expand launches + insert, over the sum of rank 0's kernel
        # times in the profiled pass.  Forwarded parents received ~ forwarded parents sent (16 B each over NVLink).
        hbm, how = measured_peaks()
        n_, P_ = len(seqs), len(seqs) * (len(seqs) - 1) // 2
        cnt, kms = r_main["rank0_counts_per_step"], r_main["rank0_kernel_ms_per_step"]
        fwd = r_main["nvlink_bytes_per_step_per_gpu"] / 16.0 if r_main["forward"] else 0.0
        alg = (cnt["pops"] * 20.0 + cnt["expansions"] * 16.0 + (cnt["expansions"] + fwd) * (16.0 + n_ + 16 * P_) + cnt["probed"] * 32.0
               + cnt["survivors"] * 24.0 + cnt["survivors"] * 56.0 + cnt["pushed"] * 36.0)
        tms = sum(kms.values())
        line["roofline"] = {"bound": "hbm", "kernel": "search round on rank 0: claim + expand (own parents) + expand (forwarded parents) + insert",
                            "achieved": alg / (tms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": alg / (tms * 1e-3) / 1e9 / hbm, "traffic": None,
                            "peak_source": how, "algorithmic_bytes_per_launch": alg, "kernel_ms_per_step": tms,
                            "note": "per-kernel roofline and ncu traffic: the N = 1 line (profiles/r02_bench_n1.json); cpu_baseline is reported at N = 1 only"}
    if world == 1:
        hbm, how = measured_peaks()
        P, S, n = G.npairs, G.S, G.n
        # algorithmic bytes per kernel of the round (DESIGN.md §4).  claim: per pop the open-list slot (4) + the table
        # entry (16), per live parent its compacted record (16).  expand+probe: per expansion the parent record (16) +
        # residues (N) + 4 cells per pair (16 P), per probed successor one 32 B table sector, per survivor its record
        # (24).  insert: per survivor the record (24) + its table sector (32); per pushed node the sector written back
        # (32) + its open-list slot (4).
        surv = c1.get("survivors", 0) - c0.get("survivors", 0) if "survivors" in c1 else None
        n_surv = surv if surv else d["pushed"]  # lower bound when the library does not count survivors
        kern = {
            "select_kernel": (select_ms, 0.0),
            "claim_kernel<1,4>": (claim_ms, d["pops"] * 20.0 + d["expansions"] * 16.0),
            "expand_probe_kernel<7,1,4,0>": (expand_ms, d["expansions"] * (16.0 + n + 16 * P) + d["probed"] * 32.0 + n_surv * 24.0),
            "insert_kernel<1,4>": (insert_ms, n_surv * 56.0 + d["pushed"] * 36.0),
        }
        allk = {}
        for name, (kms, alg) in kern.items():
            allk[name] = {"ms_per_step": kms / K, "share_of_step": kms / ms, "algorithmic_bytes_per_launch": alg / K,
                          "achieved_gbs": (alg / (kms * 1e-3) / 1e9) if kms > 0 else None}
        top = max((k for k in kern if k != "select_kernel"), key=lambda k: kern[k][0])
        tms, alg = kern[top]
        achieved = alg / (tms * 1e-3) / 1e9
        line["roofline"] = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": hbm, "unit": "GB/s",
                            "frac": achieved / hbm, "traffic": None, "peak_source": how, "launches": K,
                            "avg_launch_us": 1e3 * tms / K, "algorithmic_bytes_per_launch": alg / K,
                            "share_of_step": tms / ms, "kernels": allk,
                            "whole_round_frac": sum(v[1] for v in kern.values()) / (ms * 1e-3) / 1e9 / hbm}
        # DRAM bytes per launch of the same kernel from one `ncu --set full` capture of this workload (tools/ncu_round.sh;
        # summaries under profiles/): null when no capture of the current kernel is recorded
        tr = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tr):
            try:
                t_ = json.load(open(tr))
                line["roofline"]["traffic"] = t_["kernels"].get(top.split("<")[0])
                line["roofline"]["traffic_source"] = t_.get("source")
            except Exception:
                pass
        if args.quick:  # kernel-tuning runs: the round's timing only
            line["extra"] = {"quick": True}
            print(json.dumps(line), flush=True)
            G.close()
            return
        # ---- pairwise DP and stand-alone expansion kernel (the other two headline kernels)
        st = stream.cuda_stream
        Kx = 100000
        rng = np.random.default_rng(1)
        pos = np.stack([rng.integers(0, LENGTH, Kx) for _ in range(n)], axis=1).astype(np.uint16)
        nodes = G.make_nodes(pos, rng.integers(0, 100000, Kx), rng.integers(1, 1 << n, Kx))
        d_par = torch.from_numpy(nodes.view(np.uint8).reshape(Kx, -1)).cuda()
        sst = m.succ_dtype(n).itemsize
        d_out = torch.empty(Kx * S * sst, dtype=torch.uint8, device="cuda")
        d_cnt = torch.empty(Kx, dtype=torch.int32, device="cuda")
        for _ in range(3):
            G.expand_batch_dev(d_par.data_ptr(), Kx, 8, d_out.data_ptr(), d_cnt.data_ptr(), st)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(10):
            G.expand_batch_dev(d_par.data_ptr(), Kx, 8, d_out.data_ptr(), d_cnt.data_ptr(), st)
        a1.record(stream)
        torch.cuda.synchronize()
        xms = a0.elapsed_time(a1) / 10
        bexp = m.node_dtype(n).itemsize + n + 16 * P + S * sst  # SURVEY §8d: 4435 B at N=7
        extra["expand_only"] = {"kernel": "expand_batch_kernel<7>", "expansions_per_sec": Kx / (xms * 1e-3), "successors_per_sec": Kx * S / (xms * 1e-3),
                                "bytes_per_expansion": bexp, "achieved_gbs": Kx * bexp / (xms * 1e-3) / 1e9,
                                "frac_of_hbm": Kx * bexp / (xms * 1e-3) / 1e9 / hbm, "output_mb": Kx * S * sst / 1e6}
        try:
            gl = m.bench_random_gather(cap * 16, local)
            probes = d["probed"] / (expand_ms * 1e-3)
            extra["gather_roofline"] = {"what": "random 16 B loads/s over a table of the bench's size, 8 in flight per thread (pg_bench_random_gather)",
                                        "table_gib": cap * 16 / 2**30, "measured_loads_per_sec": gl, "kernel_probes_per_sec": probes,
                                        "frac": probes / gl}
        except Exception as ex:
            extra["gather_roofline"] = {"error": repr(ex)}
        # integer peak for the DP, two ways: (a) measured - a kernel that issues only the DP cell's own arithmetic (3 adds +
        # min3, 8 independent chains per thread) on every SM; (b) nominal lanes x clock at the 8 thread instructions per
        # cell the DP kernel actually executes (staging, shuffles, stores included)
        try:
            cell_peak_gcups = m.bench_int_peak(local) / 1e9
        except Exception:
            cell_peak_gcups = None
        int_peak_gcups = 148 * 128 * (clocks.get("sm_mhz") or 1965) * 1e6 / 8 / 1e9  # linear-gap kernel: ~118 warp instructions per 16-cell block + staging
        extra["pair_dp"] = {"kernel": "pair_dp_kernel", "cells": cells, "ms": dp_ms, "gcups": cells / (dp_ms * 1e-3) / 1e9,
                            "frac_of_integer_peak": cells / (dp_ms * 1e-3) / 1e9 / int_peak_gcups,
                            "integer_peak_gcups": int_peak_gcups, "measured_cell_arithmetic_peak_gcups": cell_peak_gcups,
                            "frac_of_measured_cell_peak": (cells / (dp_ms * 1e-3) / 1e9 / cell_peak_gcups) if cell_peak_gcups else None,
                            "note": "latency-bound wavefront, one CTA per pair: 21 of 148 SMs busy; bound by the L1 + L2 - 1 anti-diagonal steps, not by the integer pipes"}
        # ---- BASELINE configs[4]: synthetic 8 x 1000 - the 28-table heuristic build and the batched expansion at N = 8
        try:
            import random
            r8 = random.Random(SEED)
            seqs8 = ["".join(r8.choice(AA) for _ in range(1000)) for _ in range(8)]
            G8 = m.PastarGPU(seqs8, device=local)
            G8.set_stream(stream.cuda_stream)
            dp8 = min(G8.build_pair_tables() for _ in range(3))
            cells8 = sum((len(a) + 1) * (len(b) + 1) for i, a in enumerate(seqs8) for b in seqs8[i + 1:])
            K8 = 50000
            pos8 = np.stack([rng.integers(0, 1000, K8) for _ in range(8)], axis=1).astype(np.uint16)
            nodes8 = G8.make_nodes(pos8, rng.integers(0, 100000, K8), rng.integers(1, 256, K8))
            d_par8 = torch.from_numpy(nodes8.view(np.uint8).reshape(K8, -1)).cuda()
            sst8 = m.succ_dtype(8).itemsize
            d_out8 = torch.empty(K8 * 255 * sst8, dtype=torch.uint8, device="cuda")
            d_cnt8 = torch.empty(K8, dtype=torch.int32, device="cuda")
            for _ in range(3):
                G8.expand_batch_dev(d_par8.data_ptr(), K8, 8, d_out8.data_ptr(), d_cnt8.data_ptr(), st)
            torch.cuda.synchronize()
            a0.record(stream)
            for _ in range(10):
                G8.expand_batch_dev(d_par8.data_ptr(), K8, 8, d_out8.data_ptr(), d_cnt8.data_ptr(), st)
            a1.record(stream)
            torch.cuda.synchronize()
            x8 = a0.elapsed_time(a1) / 10
            b8 = m.node_dtype(8).itemsize + 8 + 16 * 28 + 255 * sst8  # SURVEY 8d: 8644 B at N=8
            extra["s8"] = {"workload": "synthetic N=8 x L=1000 (seed %d)" % SEED,
                           "pair_dp": {"tables": 28, "cells": cells8, "ms": dp8, "gcups": cells8 / (dp8 * 1e-3) / 1e9,
                                       "frac_of_integer_peak": cells8 / (dp8 * 1e-3) / 1e9 / int_peak_gcups,
                                       "frac_of_measured_cell_peak": (cells8 / (dp8 * 1e-3) / 1e9 / cell_peak_gcups) if cell_peak_gcups else None},
                           "expand_only": {"kernel": "expand_batch_kernel<8>", "expansions_per_sec": K8 / (x8 * 1e-3),
                                           "successors_per_sec": K8 * 255 / (x8 * 1e-3), "bytes_per_expansion": b8,
                                           "achieved_gbs": K8 * b8 / (x8 * 1e-3) / 1e9, "frac_of_hbm": K8 * b8 / (x8 * 1e-3) / 1e9 / hbm}}
            del d_out8
            G8.close()
        except Exception as ex:
            extra["s8"] = {"error": repr(ex)}
        del d_out

        # ---- e2e: host buffers -> C ABI -> result.  The job is 4x the expansions of ramp-up + warm-up + timed region, so
        # that the one-off set-up (context, 16 GiB table allocation and clear) does not dominate a sub-second search.
        torch.cuda.synchronize()
        r, wall, t_ctx, factor = None, 0.0, 0.0, 4.0  # the untimed-arm ramp-up (small frontiers) is part of this job: a longer job amortises it
        while r is None:
            budget = int(factor * c1["expansions"])
            t0 = time.perf_counter()
            G2 = m.PastarGPU(seqs, device=local)          # host weights + H2D of residues / cost table / weights
            t_ctx = time.perf_counter() - t0
            G2.build_pair_tables()
            try:
                r = G2.search(table_capacity=cap, batch_target=batch, max_expansions=budget, want_rows=False)
            except m.PastarError:
                if factor <= 1.0:
                    raise
                factor = 1.0                              # table / pool too small for the longer job: the timed arm's own length
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            G2.close()
        h2d = sum(((len(s) + 16) & ~15) for s in seqs) + 8100 * 4 + 2 * n + 16
        d2h = (r["rounds"] // 8 + 2) * 200 + 16
        line["e2e"] = {"value": r["expansions"] / wall, "unit": UNIT, "h2d_bytes_per_step": h2d / max(1, r["rounds"]),
                       "d2h_bytes_per_step": d2h / max(1, r["rounds"]), "expansions": r["expansions"], "rounds": r["rounds"],
                       "wall_s": wall, "context_s": t_ctx, "search_kernel_s": r["kernel_ms"] * 1e-3,
                       "includes": "host Altschul weights, context create, pairwise DP, table set-up (16 GiB of value blocks cleared; the buffers themselves come from the library's cache of the timed arm's search, as in any second job of a process), search from the start node "
                                   "(%.1fx the expansions of the timed arm's whole run), result read-back" % factor}
        # ---- a TERMINATING anchor: kinase.fasta (BASELINE configs[1]) solved to the optimality-preserving stop, on the device
        # and end to end from host buffers; expansions raw and "useful" (no more than the serial A* needs: batching expands
        # nodes a serial search never would, SURVEY 7)
        try:
            kseqs = PARITY_INPUTS["kinase"][0]
            t0 = time.perf_counter()
            Gk = m.PastarGPU(kseqs, device=local)
            Gk.build_pair_tables()
            rk = Gk.search(table_capacity=1 << 26, batch_target=16384, want_rows=True)
            torch.cuda.synchronize()
            wall_k = time.perf_counter() - t0
            ok_k = rk["finished"] == 1 and rk["g"] == 421546 and m.rescore_alignment(kseqs, Gk.w_int, rk["rows"]) == 421546
            Gk.close()
            serial = 4497278  # expansions of the serial A* on the reference's arithmetic (oracle/_ref astar; tie-break dependent)
            extra["kinase"] = {"workload": "kinase.fasta (5 x 263-276) full solve, batch 16384", "optimal_cost": rk["g"], "parity": "ok" if ok_k else "FAILED",
                               "expansions_raw": rk["expansions"], "expansions_useful": min(rk["expansions"], serial), "serial_astar_expansions": serial,
                               "rounds": rk["rounds"], "device_ms": rk["kernel_ms"], "value_expansions_per_sec": rk["expansions"] / (rk["kernel_ms"] * 1e-3),
                               "useful_expansions_per_sec": min(rk["expansions"], serial) / (rk["kernel_ms"] * 1e-3),
                               "e2e_wall_s": wall_k, "e2e_expansions_per_sec": rk["expansions"] / wall_k,
                               "cpu_reference_full_solve": {"seconds": 398.0, "threads": 1, "what": "oracle/_ref serial A* (AStar.cpp:53-104 semantics) on the survey container, recorded in DESIGN.md; not re-run here (bounded bench)"}}
            if not ok_k:
                raise SystemExit("kinase.fasta: optimal cost / alignment mismatch")
            try:  # the CPU path on the same input, bounded to ~10 s
                from oracle import refio
                if refio.available():
                    threads = os.cpu_count() or 1
                    rc_ = refio.pastar(kseqs, threads, 400000, "FZORDER", 12, timeout=600, warm_pops=20000)
                    extra["kinase"]["cpu_reference_sample"] = {"expansions_per_sec": rc_["timed_expansions"] / rc_["timed_seconds"], "threads": threads,
                                                               "dequeues": 400000, "kind": "reference"}
            except Exception as ex:
                extra["kinase"]["cpu_reference_sample"] = {"error": repr(ex)}
        except SystemExit:
            raise
        except Exception as ex:
            extra["kinase"] = {"error": repr(ex)}
        # ---- CPU baseline beside it (bounded sample)
        try:
            threads = os.cpu_count() or 1
            b = cpu_reference_run(threads, 100, 10)  # 1.5 M dequeues after 150 K warm-up: 10-30 s of CPU work
            line["cpu_baseline"] = {k: b[k] for k in ("value", "unit", "cores", "kind", "sample")}
            try:
                line["cpu_baseline"]["micro"] = cpu_micro_baselines()
            except Exception as ex:
                line["cpu_baseline"]["micro"] = {"error": repr(ex)}
        except Exception as ex:  # never lose the GPU numbers to a CPU-side hiccup
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}
    else:
        # ---- e2e at N GPUs: the whole job through the public multi-GPU API (mpi_pastar_msa_b200.dist over the C ABI) from
        # host buffers: per rank host weights, context create, pairwise DP, engine set-up (peer-mapped inboxes), the
        # search from the start node budgeted to the expansions the timed arm did in total, status read-backs.
        # As at N = 1 the job is 4x the expansions of the timed arm's whole run (ramp-up + warm-up + timed rounds), so that
        # the one-off set-up does not dominate a sub-second search; 1x if the table cannot hold the longer job.
        G.close()
        # (capped at ~200 M expansions per GPU: what a 2^30-slot table holds with room to spare)
        r, wall, factor = None, 0.0, max(1.0, min(4.0, 200e6 * world / max(1, tot1[0])))
        while r is None:
            budget = int(factor * tot1[0])
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            G2 = m.PastarGPU(seqs, device=local)
            G2.set_stream(stream.cuda_stream)
            G2.build_pair_tables()
            eng2, _ = make_engine(G2, args.hash_type, args.hash_shift)
            drv2 = PartitionedSearch(eng2, dist, seqs, lambda pos: int(G2.owner(np.array(pos, dtype=np.uint16), world)[0]), max_expansions=budget)
            drv2.rounds_per_status = 8
            failed = torch.zeros(1, dtype=torch.int64, device="cuda")
            try:
                r = drv2.run()
            except m.PastarError:
                failed += 1
            dist.all_reduce(failed)  # every rank takes the same branch
            torch.cuda.synchronize()
            dist.barrier()
            wall = time.perf_counter() - t0
            eng2.end()
            G2.close()
            if int(failed.item()):
                if factor <= 1.0:
                    raise SystemExit("e2e job failed at N = %d" % world)
                r, factor = None, 1.0
        h2d = sum(((len(s) + 16) & ~15) for s in seqs) + 8100 * 4 + 2 * len(seqs) + 16
        n_status = r["rounds"] // 8 + 2
        line["e2e"] = {"value": r["expansions"] / wall, "unit": UNIT, "h2d_bytes_per_step": world * (h2d + 40 * n_status) / max(1, r["rounds"]),
                       "d2h_bytes_per_step": world * (n_status * (160 + 40 * world)) / max(1, r["rounds"]), "expansions": r["expansions"],
                       "rounds": r["rounds"], "wall_s": wall,
                       "includes": "per rank: host Altschul weights, context create, pairwise DP, P2P engine set-up (table buffers and peer-mapped inboxes reused from the caches the timed arm filled, cleared), the partitioned search "
                                   "from the start node (PartitionedSearch.run, %.1fx the expansions of the timed arm's whole run), one status exchange every 8 rounds" % factor}
    if parity is not None:
        line["parity"] = parity
    line["extra"] = extra
    if world == 1:
        G.close()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="open-list entries popped per round and GPU")
    ap.add_argument("--table-capacity", type=int, default=1 << 30)
    ap.add_argument("--quick", action="store_true", help="N = 1: print the round's timing only (no extras, e2e or CPU baseline)")
    ap.add_argument("--skip-parity", action="store_true", help="N > 1: skip the untimed PF08184 / kinase parity gate (profiling runs)")
    ap.add_argument("--hash-type", default="PZORDER", choices=["FZORDER", "PZORDER", "FSUM", "PSUM"],
                    help="owner hash for N > 1 (the reference's -y; its default FZORDER shift 12 is reported in extra.owner_hash_sweep)")
    ap.add_argument("--hash-shift", type=int, default=6,
                    help="owner-hash shift for N > 1 (the reference's -s, 0..21).  PZORDER shift 6 takes bits 3-4 of the first two "
                         "coordinates: an eighth of the parents straddle a partition boundary per owner coordinate; FZORDER shift 12 "
                         "(bit 1 of five coordinates) makes most parents straddle several")
    ap.add_argument("--no-hash-sweep", action="store_true", help="N > 1: skip the FZORDER shift 12 / 17 comparison runs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N = 1: write what the timed rounds computed as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
