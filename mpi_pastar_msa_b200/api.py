"""ctypes binding of libpastar_gpu.so, shaped like the reference's interfaces.

Reference interface                                   -> here
  read_fasta_file (pastar/read_fasta.cpp:8-36)         -> read_fasta
  Sequences::set_seq + HeuristicHPair::init            -> PastarGPU(seqs) + .build_pair_tables()
     (Sequences.cpp:39-51, HeuristicHPair.cpp:47-67)
  PairAlign::getScore (PairAlign.cpp:174-177)          -> .pair_table(pair)[i, j]
  HeuristicHPair::calculate_h (HeuristicHPair.cpp:73)  -> .calculate_h(coords)
  Coord::configure_hash / get_id (CoordHash.cpp)       -> .configure_hash / .owner
  Node::getNeigh (Node.cpp:205-248)                    -> .expand_batch / .get_neigh
  PAStar::pa_star (PAStar.cpp:626-673)                 -> .search
  (no reference counterpart: bounded-suboptimal search) -> .search(weight=W) / .search_set_weight / .search_lower_bound
  (no reference counterpart: incumbent / anytime search) -> .score_alignment / .search(incumbent=rows) / .anytime_search
"""
import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
HASH_TYPES = {"FZORDER": 0, "PZORDER": 1, "FSUM": 2, "PSUM": 3}
_STATUS = {1: "PG_ERR_ARG", 2: "PG_ERR_CUDA", 3: "PG_ERR_UNSUPPORTED", 4: "PG_ERR_CAPACITY", 5: "PG_ERR_STATE",
           6: "PG_ERR_HASH_SHIFT"}
SUPPORTED_N = (3, 4, 5, 6, 7, 8, 9, 10, 14, 16)  # max_seq_helper.h:9-19


class PastarError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (_STATUS.get(code, code), msg))
        self.code = code


class SearchConfig(C.Structure):
    _fields_ = [("n_parts", C.c_int32), ("part", C.c_int32), ("table_capacity", C.c_int64), ("batch_target", C.c_int64),
                ("max_expansions", C.c_int64), ("rounds_per_sync", C.c_int32), ("reserved", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("finished", C.c_int32), ("g", C.c_int32), ("f", C.c_int32), ("align_len", C.c_int32), ("pops", C.c_int64),
                ("expansions", C.c_int64), ("generated", C.c_int64), ("reopen", C.c_int64), ("open_size", C.c_int64),
                ("closed_size", C.c_int64), ("rounds", C.c_int64), ("probed", C.c_int64), ("pushed", C.c_int64),
                ("inserted", C.c_int64), ("seconds", C.c_double), ("kernel_ms", C.c_double), ("expand_ms", C.c_double),
                ("select_ms", C.c_double), ("claim_ms", C.c_double), ("insert_ms", C.c_double),
                ("survivors", C.c_int64), ("inbox_ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def lib_path():
    # PASTAR_GPU_LIB selects another build of the same library (e.g. one compiled with -DPG_PHASE_TIMING)
    return os.environ.get("PASTAR_GPU_LIB") or os.path.join(_HERE, "lib", "libpastar_gpu.so")


_lib = None


def load_library():
    """Load libpastar_gpu.so.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise PastarError(2, "libpastar_gpu.so is not built (python -m mpi_pastar_msa_b200.build); no CPU fallback exists")
    L = C.CDLL(p)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    sig = {
        "pg_abi_version": ([], i32),
        "pg_last_error": ([vp], C.c_char_p),
        "pg_default_cost_table": ([vp], None),
        "pg_host_weights": ([i32, C.POINTER(C.c_char_p), C.POINTER(i32), vp], i32),
        "pg_gpu_weights": ([i32, C.POINTER(C.c_char_p), C.POINTER(i32), i32, vp, C.POINTER(C.c_float)], i32),
        "pg_ctx_create": ([i32, C.POINTER(C.c_char_p), C.POINTER(i32), vp, i32, i32, i32, vp, i32, C.POINTER(vp)], i32),
        "pg_ctx_destroy": ([vp], None),
        "pg_allow_extended_n": ([i32], i32),
        "pg_ctx_set_stream": ([vp, vp], i32),
        "pg_search_rounds": ([vp, C.c_int32, C.c_int32], i32),
        "pg_search_profile": ([vp, i32], i32),
        "pg_search_note_rounds": ([vp, C.c_int64], i32),
        "pg_release_cached_memory": ([], None),
        "pg_build_pair_tables": ([vp, C.POINTER(C.c_float)], i32),
        "pg_pair_table_shape": ([vp, i32, C.POINTER(i32), C.POINTER(i32)], i32),
        "pg_copy_pair_table": ([vp, i32, vp], i32),
        "pg_calculate_h": ([vp, vp, i64, vp], i32),
        "pg_configure_hash": ([vp, i32, i32], i32),
        "pg_owner": ([vp, vp, i64, i32, vp], i32),
        "pg_expand_batch": ([vp, vp, i64, i32, vp, vp], i32),
        "pg_expand_batch_dev": ([vp, vp, i64, i32, vp, vp, vp], i32),
        "pg_search": ([vp, C.POINTER(SearchConfig), C.POINTER(Result), C.POINTER(C.c_char_p)], i32),
        "pg_search_begin": ([vp, C.POINTER(SearchConfig)], i32),
        "pg_search_round": ([vp, C.c_int32], i32),
        "pg_search_outbox": ([vp, i32, C.POINTER(vp), C.POINTER(i64)], i32),
        "pg_search_insert_dev": ([vp, vp, i64], i32),
        "pg_bench_random_gather": ([i32, i64, C.POINTER(C.c_double)], i32),
        "pg_bench_int_peak": ([i32, C.POINTER(C.c_double)], i32),
        "pg_search_set_peers": ([vp, C.POINTER(vp), i32], i32),
        "pg_search_set_peer_counts": ([vp, C.POINTER(vp), i32, i32], i32),
        "pg_search_round_async": ([vp, C.c_int32], i32),
        "pg_search_set_device_sync": ([vp, i32], i32),
        "pg_search_insert_inbox_async": ([vp], i32),
        "pg_search_sync": ([vp], i32),
        "pg_multi_search": ([C.POINTER(vp), i32, C.POINTER(SearchConfig), C.POINTER(Result), C.POINTER(Result), C.POINTER(C.c_char_p)], i32),
        "pg_search_region_bytes": ([vp], i64),
        "pg_search_outbox_capacity": ([vp], i64),
        "pg_search_outbox_counts_dev": ([vp, C.POINTER(vp)], i32),
        "pg_search_insert_segments_dev": ([vp, vp, i64, C.POINTER(i64), i32], i32),
        "pg_search_status": ([vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(Result)], i32),
        "pg_search_lookup": ([vp, vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)], i32),
        "pg_search_end": ([vp], i32),
        "pg_xrec_stride": ([vp], i32),
        "pg_search_set_weight": ([vp, C.c_int32, C.c_int32], i32),
        "pg_search_lower_bound": ([vp, C.POINTER(C.c_int32)], i32),
        "pg_score_alignment": ([vp, C.POINTER(C.c_char_p), C.c_int32, C.POINTER(C.c_int64)], i32),
        "pg_search_set_incumbent": ([vp, C.POINTER(C.c_char_p), C.c_int32], i32),
        "pg_search_anytime": ([vp, C.POINTER(SearchConfig), C.POINTER(C.c_int32), C.POINTER(C.c_int32), i32, C.POINTER(Result),
                               C.POINTER(Result), C.POINTER(C.c_int32), C.POINTER(C.c_char_p)], i32),
    }
    for name, (args, res) in sig.items():
        f = getattr(L, name)
        f.argtypes = args
        f.restype = res
    _lib = L
    return L


EXPORTS = ["pg_release_cached_memory", "pg_search_note_rounds", "pg_search_set_device_sync", "pg_allow_extended_n", "pg_gpu_weights", "pg_bench_int_peak", "pg_multi_search", "pg_search_region_bytes", "pg_search_set_peer_counts", "pg_search_round_async", "pg_search_insert_inbox_async", "pg_search_sync", "pg_bench_random_gather", "pg_search_set_peers", "pg_search_outbox_capacity", "pg_search_outbox_counts_dev", "pg_search_insert_segments_dev",
           "pg_ctx_set_stream", "pg_search_rounds", "pg_search_profile", "pg_abi_version", "pg_last_error", "pg_default_cost_table", "pg_host_weights", "pg_ctx_create", "pg_ctx_destroy",
           "pg_build_pair_tables", "pg_pair_table_shape", "pg_copy_pair_table", "pg_calculate_h", "pg_configure_hash",
           "pg_owner", "pg_expand_batch", "pg_expand_batch_dev", "pg_search", "pg_search_begin", "pg_search_round",
           "pg_search_outbox", "pg_search_insert_dev", "pg_search_status", "pg_search_lookup", "pg_search_end",
           "pg_xrec_stride", "pg_search_set_weight", "pg_search_lower_bound", "pg_score_alignment", "pg_search_set_incumbent",
           "pg_search_anytime"]

WEIGHT_DEN = 1024


def weight_fraction(weight):
    """Search weight W (1 <= W <= 16) as (num, den): num / 1024 rounded up, as the pastar CLI's --weight."""
    return int(math.ceil(float(weight) * WEIGHT_DEN)), WEIGHT_DEN


def node_dtype(n):
    """Node<N> record (Node.h:28-49): uint16 pos[N], pad to 4, int32 f, g, parenti."""
    base = (2 * n + 3) & ~3
    return np.dtype({"names": ["pos", "f", "g", "parenti"], "formats": [("<u2", (n,)), "<i4", "<i4", "<i4"],
                     "offsets": [0, base, base + 4, base + 8], "itemsize": base + 12})


def succ_dtype(n):
    """Node<N> + uint32 owner (= Coord<N>::get_id(vec_size))."""
    base = (2 * n + 3) & ~3
    return np.dtype({"names": ["pos", "f", "g", "parenti", "owner"], "formats": [("<u2", (n,)), "<i4", "<i4", "<i4", "<u4"],
                     "offsets": [0, base, base + 4, base + 8, base + 12], "itemsize": base + 16})


def read_fasta(path):
    """read_fasta_file_core (pastar/read_fasta.cpp:8-36): '>' lines and empty lines end a record; no validation."""
    seqs, cur = [], ""
    with open(path) as f:
        for line in f.read().split("\n"):
            if len(line) == 0 or line[0] == ">":
                if cur:
                    seqs.append(cur)
                cur = ""
            else:
                cur += line
    if cur:
        seqs.append(cur)
    return seqs


def _seq_args(seqs):
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    return bs, (C.c_char_p * len(bs))(*bs), (C.c_int * len(bs))(*[len(b) for b in bs])


def default_cost_table():
    out = np.zeros(8100, dtype=np.int32)
    load_library().pg_default_cost_table(out.ctypes.data)
    return out.reshape(90, 90)


def bench_random_gather(nbytes, device=-1):
    """Random 16-byte loads/s over an nbytes table: the measured ceiling for the dedupe probe."""
    out = C.c_double()
    rc = load_library().pg_bench_random_gather(device, int(nbytes), C.byref(out))
    if rc:
        raise PastarError(rc, "pg_bench_random_gather")
    return out.value


def multi_search(gpus, table_capacity=0, batch_target=0, max_expansions=0, rounds_per_sync=0, want_rows=True, weight=1.0,
                 incumbent=None):
    """pg_multi_search: one hash-owned partition per context in `gpus` (PastarGPU objects with their pair tables built and
    the same hash configuration; normally one per device, but contexts on one device work too), driven by this process.
    weight != 1: bounded-suboptimal search (see PastarGPU.search), set on every context.
    incumbent (alignment rows): set on every context (see PastarGPU.search).
    Returns (total dict with lower_bound / weight_num / weight_den, list of per-partition dicts)."""
    L = load_library()
    g0 = gpus[0]
    if weight != 1.0:
        for g in gpus:
            g.search_set_weight(*weight_fraction(weight))
    if incumbent is not None:
        for g in gpus:
            g.search_set_incumbent(incumbent)
    cfg = SearchConfig(len(gpus), 0, table_capacity, batch_target, max_expansions, rounds_per_sync, 0)
    res, parts = Result(), (Result * len(gpus))()
    handles = (C.c_void_p * len(gpus))(*[g.h for g in gpus])
    rows, bufs = g0._row_bufs(want_rows)
    g0._ck(L.pg_multi_search(handles, len(gpus), C.byref(cfg), C.byref(res), parts, rows))
    d = g0._result(res, bufs)
    d["weight_num"], d["weight_den"] = g0.weight
    return d, [p.as_dict() for p in parts]


def rescore_alignment(seqs, w_int, rows, cost=None, gap_open=30, gap_ext=30, gap_gap=30):
    """Host-side self check: the g of the path an alignment describes under the reference's cost model (Node.cpp:129-152,
    240-243; weights (int)weightMatrix[x][y]).  A search result is valid iff its rows spell the sequences and re-score
    to the reported optimum."""
    cost = default_cost_table() if cost is None else np.asarray(cost).reshape(90, 90)
    n, cols = len(seqs), len(rows[0])
    if any(len(r) != cols for r in rows) or any(rows[i].replace("-", "") != seqs[i] for i in range(n)):
        raise ValueError("alignment rows do not spell the input sequences")
    prev, total = [1] * n, 0  # initial parenti: all ones (Sequences.cpp:75)
    for c in range(cols):
        mv = [0 if rows[i][c] == "-" else 1 for i in range(n)]
        if not any(mv):
            raise ValueError("empty alignment column")
        for x in range(n - 1):
            for y in range(x + 1, n):
                if mv[x] and mv[y]:
                    t = int(cost[ord(rows[x][c]), ord(rows[y][c])])
                elif mv[x] or mv[y]:
                    s = y if mv[x] else x          # the sequence that takes the gap
                    t = gap_open if prev[s] else gap_ext
                else:
                    t = gap_gap
                total += t * int(w_int[x][y])
        prev = mv
    return total


def bench_int_peak(device=-1):
    """DP-cell instruction groups (3 adds + min3) per second the integer pipes sustain: the pairwise DP's measured peak."""
    out = C.c_double()
    rc = load_library().pg_bench_int_peak(device, C.byref(out))
    if rc:
        raise PastarError(rc, "pg_bench_int_peak")
    return out.value


def host_weights(seqs):
    """weightAltschulsRationale2 (WeightedSP.cpp:424-519): float32 n x n, computed on the host."""
    _, arr, lens = _seq_args(seqs)
    n = len(seqs)
    out = np.zeros((n, n), dtype=np.float32)
    rc = load_library().pg_host_weights(n, arr, lens, out.ctypes.data)
    if rc:
        raise PastarError(rc, "pg_host_weights")
    return out


def release_cached_memory():
    """Give the device buffers the library keeps between searches back to the driver (pg_release_cached_memory)."""
    load_library().pg_release_cached_memory()


def allow_extended_n(enable=True):
    """Explicit opt-in (diverges from the reference, max_seq_helper.h:9-19): also accept N = 11, 12, 13, 15 on one GPU."""
    load_library().pg_allow_extended_n(1 if enable else 0)


def gpu_weights(seqs, device=-1, want_ms=False):
    """weightAltschulsRationale2 with the pair loop (primer, WeightedSP.cpp:144-244) as one kernel: same floats as host_weights."""
    L = load_library()
    n = len(seqs)
    keep = _seq_args(seqs)
    out = np.zeros((n, n), dtype=np.float32)
    ms = C.c_float(0)
    rc = L.pg_gpu_weights(n, keep[1], keep[2], device, out.ctypes.data, C.byref(ms))
    if rc:
        raise PastarError(rc, "pg_gpu_weights failed")
    return (out, ms.value) if want_ms else out


class PastarGPU:
    """One problem (sequence set) on one GPU: the Sequences + Cost + HeuristicHPair singletons of the reference."""

    def __init__(self, seqs, weights="altschul", cost=None, gap_open=30, gap_ext=30, gap_gap=30, device=-1):
        self.L = load_library()
        self.seqs = [s if isinstance(s, str) else s.decode() for s in seqs]
        self.n = len(self.seqs)
        self.lens = [len(s) for s in self.seqs]
        self.npairs = self.n * (self.n - 1) // 2
        self.S = (1 << self.n) - 1
        if isinstance(weights, str) and weights in ("altschul", "altschul_host"):
            # pair loop of the weight routine on the device (pg_gpu_weights); the host routine for sequences beyond its
            # shared-memory sweep or on request - both give the reference's floats bit for bit
            self.weights_f = None
            if weights == "altschul":
                try:
                    self.weights_f = gpu_weights(self.seqs, device)
                except PastarError as e:
                    if e.code != 3:
                        raise
            if self.weights_f is None:
                self.weights_f = host_weights(self.seqs)
            self.w_int = self.weights_f.astype(np.int32)  # (int) truncation, Node.cpp:226
        elif weights is None:
            self.weights_f, self.w_int = None, np.ones((self.n, self.n), dtype=np.int32)
        else:
            self.weights_f, self.w_int = None, np.ascontiguousarray(weights, dtype=np.int32).reshape(self.n, self.n)
        self._keep = _seq_args(self.seqs)
        costp = None
        if cost is not None:
            self._cost = np.ascontiguousarray(cost, dtype=np.int32).reshape(8100)
            costp = self._cost.ctypes.data
        h = C.c_void_p()
        rc = self.L.pg_ctx_create(self.n, self._keep[1], self._keep[2], costp, gap_open, gap_ext, gap_gap,
                                  self.w_int.ctypes.data, device, C.byref(h))
        self.h = h
        if rc:
            msg = self.L.pg_last_error(h).decode() if h else "pg_ctx_create"
            if h:
                self.L.pg_ctx_destroy(h)
                self.h = None
            raise PastarError(rc, msg)
        self.tables_ms = None
        self.weight = (1, 1)  # (num, den) of the search weight last set on the context

    def close(self):
        if getattr(self, "h", None):
            self.L.pg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc:
            raise PastarError(rc, self.L.pg_last_error(self.h).decode())

    # ---- (1) heuristic
    def build_pair_tables(self):
        ms = C.c_float()
        self._ck(self.L.pg_build_pair_tables(self.h, C.byref(ms)))
        self.tables_ms = ms.value
        return ms.value

    def pair_table(self, pair):
        r, c = C.c_int(), C.c_int()
        self._ck(self.L.pg_pair_table_shape(self.h, pair, C.byref(r), C.byref(c)))
        out = np.zeros((r.value, c.value), dtype=np.int32)
        self._ck(self.L.pg_copy_pair_table(self.h, pair, out.ctypes.data))
        return out

    def calculate_h(self, coords):
        a = np.ascontiguousarray(coords, dtype=np.uint16).reshape(-1, self.n)
        out = np.zeros(a.shape[0], dtype=np.int32)
        self._ck(self.L.pg_calculate_h(self.h, a.ctypes.data, a.shape[0], out.ctypes.data))
        return out

    # ---- (3) owner
    def configure_hash(self, hash_type="FZORDER", shift=12):
        self._ck(self.L.pg_configure_hash(self.h, HASH_TYPES[hash_type] if isinstance(hash_type, str) else hash_type, shift))

    def owner(self, coords, size):
        a = np.ascontiguousarray(coords, dtype=np.uint16).reshape(-1, self.n)
        out = np.zeros(a.shape[0], dtype=np.uint32)
        self._ck(self.L.pg_owner(self.h, a.ctypes.data, a.shape[0], size, out.ctypes.data))
        return out

    # ---- (2) expansion
    def make_nodes(self, pos, g, parenti):
        pos = np.asarray(pos, dtype=np.uint16).reshape(-1, self.n)
        a = np.zeros(pos.shape[0], dtype=node_dtype(self.n))
        a["pos"], a["g"], a["parenti"] = pos, g, parenti
        return a

    def expand_batch(self, parents, vec_size=1):
        """Node::getNeigh for every parent.  Returns (succ[K, 2^N-1], counts[K]); row k holds counts[k] records."""
        parents = np.ascontiguousarray(parents)
        assert parents.dtype == node_dtype(self.n)
        k = parents.shape[0]
        out = np.zeros((k, self.S), dtype=succ_dtype(self.n))
        counts = np.zeros(k, dtype=np.int32)
        self._ck(self.L.pg_expand_batch(self.h, parents.ctypes.data, k, vec_size, out.ctypes.data, counts.ctypes.data))
        return out, counts

    def expand_batch_dev(self, d_parents, k, vec_size, d_out, d_counts, stream=0):
        self._ck(self.L.pg_expand_batch_dev(self.h, d_parents, k, vec_size, d_out, d_counts, stream))

    def get_neigh(self, pos, g, parenti, vec_size=1):
        """Shim of Node<N>::getNeigh(a, vec_size): a batch of one, records in the reference's order
        (bucket by owner, ascending mask inside a bucket: Node.cpp:234-246)."""
        out, counts = self.expand_batch(self.make_nodes([pos], [g], [parenti]), vec_size)
        s = out[0, :counts[0]]
        return s[np.argsort(s["owner"], kind="stable")]

    # ---- (3)+(4) search
    def _row_bufs(self, want_rows):
        if not want_rows:
            return None, None
        total = sum(self.lens) + 1
        bufs = [C.create_string_buffer(total) for _ in range(self.n)]
        return (C.c_char_p * self.n)(*[C.cast(b, C.c_char_p) for b in bufs]), bufs

    def _result(self, res, bufs):
        """A search's Result as a dict, with the rows found (when _row_bufs gave buffers) and the certified lower bound."""
        d = res.as_dict()
        if bufs is not None and res.finished:
            d["rows"] = [b.value.decode() for b in bufs]
        d["lower_bound"] = self.search_lower_bound()
        return d

    def search(self, table_capacity=0, batch_target=0, max_expansions=0, rounds_per_sync=0, want_rows=True, weight=1.0,
               incumbent=None):
        """weight W > 1: bounded-suboptimal search (num / 1024 rounded up, as the CLI's --weight): g <= W x the optimum,
        certified by the returned lower_bound (g * weight_den <= weight_num * lower_bound when finished).
        incumbent (alignment rows): set as the context's incumbent first (search_set_incumbent); finished == 2 then means
        that nothing cheaper exists below its cost (its rows and cost are returned; an exact search proves it optimal)."""
        if weight != 1.0:
            self.search_set_weight(*weight_fraction(weight))
        if incumbent is not None:
            self.search_set_incumbent(incumbent)
        cfg = SearchConfig(1, 0, table_capacity, batch_target, max_expansions, rounds_per_sync, 0)
        res = Result()
        rows, bufs = self._row_bufs(want_rows)
        self._ck(self.L.pg_search(self.h, C.byref(cfg), C.byref(res), rows))
        d = self._result(res, bufs)
        d["weight_num"], d["weight_den"] = self.weight
        return d

    def search_set_weight(self, num, den):
        """pg_search_set_weight: every later search on this context is weighted by num / den (den a power of two <= 1024,
        den <= num <= 16 den); (1, 1) is the exact search."""
        self._ck(self.L.pg_search_set_weight(self.h, int(num), int(den)))
        self.weight = (int(num), int(den))

    def _rows_arg(self, rows):
        bs = [r.encode() if isinstance(r, str) else bytes(r) for r in rows]
        if len(bs) != self.n:
            raise PastarError(1, "PG_ERR_ARG: %d alignment rows for %d sequences" % (len(bs), self.n))
        return (C.c_char_p * self.n)(*bs), len(bs[0])

    def score_alignment(self, rows):
        """pg_score_alignment: the cost of an alignment (N rows of equal length, '-' for gaps) under this context's cost
        model; PastarError PG_ERR_ARG if the rows do not align this context's sequences."""
        arr, cols = self._rows_arg(rows)
        v = C.c_int64()
        self._ck(self.L.pg_score_alignment(self.h, arr, cols, C.byref(v)))
        return v.value

    def search_set_incumbent(self, rows):
        """pg_search_set_incumbent: every later search keeps only what can beat this alignment's cost; None clears it."""
        if rows is None:
            self._ck(self.L.pg_search_set_incumbent(self.h, None, 0))
        else:
            arr, cols = self._rows_arg(rows)
            self._ck(self.L.pg_search_set_incumbent(self.h, arr, cols))

    def anytime_search(self, weights=(2, 1.25, 1), incumbent=None, table_capacity=0, batch_target=0, max_expansions=0,
                       want_rows=True):
        """pg_search_anytime: one fresh search per weight, each bounded by the best alignment so far (the incumbent, if
        given, for the first); max_expansions is the budget over all phases.  Returns the usual dict (finished 1: proved
        optimal, 2: an alignment with a gap to lower_bound, 0: none) with `lower_bound` and `phases`, one dict per phase
        that ran: weight, g, lower_bound, expansions, finished."""
        if incumbent is not None:
            self.search_set_incumbent(incumbent)
        fr = [weight_fraction(w) for w in weights]
        k = len(fr)
        nums = (C.c_int32 * k)(*[f[0] for f in fr])
        dens = (C.c_int32 * k)(*[f[1] for f in fr])
        cfg = SearchConfig(1, 0, table_capacity, batch_target, max_expansions, 0, 0)
        res, pres, plb = Result(), (Result * k)(), (C.c_int32 * k)()
        rows, bufs = self._row_bufs(want_rows)
        self._ck(self.L.pg_search_anytime(self.h, C.byref(cfg), nums, dens, k, C.byref(res), pres, plb, rows))
        d = self._result(res, bufs)
        d["phases"] = [{"weight": fr[i][0] / fr[i][1], "g": pres[i].g, "lower_bound": plb[i], "expansions": pres[i].expansions,
                        "finished": pres[i].finished} for i in range(k) if plb[i] >= 0]
        return d

    def search_lower_bound(self):
        """pg_search_lower_bound: certified lower bound on the optimal cost (of the last search, or of this partition of
        the active step-wise search)."""
        v = C.c_int32()
        self._ck(self.L.pg_search_lower_bound(self.h, C.byref(v)))
        return v.value

    # step-wise (multi-GPU drivers)
    def search_begin(self, n_parts=1, part=0, table_capacity=0, batch_target=0, p2p=False):
        """p2p: False/0 = local outboxes (NCCL all-to-all by the driver), True/1 = successor records stored into the
        owners' peer-mapped inboxes, 2 = parent forwarding over the peer-mapped inboxes."""
        cfg = SearchConfig(n_parts, part, table_capacity, batch_target, 0, 0, int(p2p))
        self._ck(self.L.pg_search_begin(self.h, C.byref(cfg)))

    def search_set_peers(self, ptrs):
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        self._ck(self.L.pg_search_set_peers(self.h, arr, len(ptrs)))

    def search_set_peer_counts(self, ptrs, nbuf=2):
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        self._ck(self.L.pg_search_set_peer_counts(self.h, arr, len(ptrs), nbuf))

    def search_set_device_sync(self, enable=True):
        self._ck(self.L.pg_search_set_device_sync(self.h, 1 if enable else 0))

    def search_round_async(self, f_limit=2**31 - 1):
        self._ck(self.L.pg_search_round_async(self.h, f_limit))

    def search_insert_inbox_async(self):
        self._ck(self.L.pg_search_insert_inbox_async(self.h))

    def search_sync(self):
        self._ck(self.L.pg_search_sync(self.h))

    def search_region_bytes(self):
        return int(self.L.pg_search_region_bytes(self.h))

    def search_outbox_capacity(self):
        return int(self.L.pg_search_outbox_capacity(self.h))

    def search_outbox_counts_dev(self):
        p = C.c_void_p()
        self._ck(self.L.pg_search_outbox_counts_dev(self.h, C.byref(p)))
        return p.value

    def search_insert_segments_dev(self, base, stride_bytes, counts):
        arr = (C.c_int64 * len(counts))(*[int(c) for c in counts])
        self._ck(self.L.pg_search_insert_segments_dev(self.h, base, stride_bytes, arr, len(counts)))

    def search_round(self, f_limit=2**31 - 1):
        self._ck(self.L.pg_search_round(self.h, f_limit))

    def search_rounds(self, rounds, f_limit=2**31 - 1):
        self._ck(self.L.pg_search_rounds(self.h, rounds, f_limit))

    def search_profile(self, enable=True):
        self._ck(self.L.pg_search_profile(self.h, 1 if enable else 0))
        self.profiling = bool(enable)

    def search_note_rounds(self, delta):
        self._ck(self.L.pg_search_note_rounds(self.h, int(delta)))

    def set_stream(self, stream):
        """cudaStream_t handle (int) the context launches on; 0 = the legacy default stream (torch's default), -1 = own."""
        self._ck(self.L.pg_ctx_set_stream(self.h, C.c_void_p(stream if stream != -1 else 2**64 - 1)))

    def search_outbox(self, dst):
        p, n = C.c_void_p(), C.c_int64()
        self._ck(self.L.pg_search_outbox(self.h, dst, C.byref(p), C.byref(n)))
        return p.value, n.value

    def search_insert_dev(self, d_records, count):
        self._ck(self.L.pg_search_insert_dev(self.h, d_records, count))

    def search_status(self):
        a, b, r = C.c_int32(), C.c_int32(), Result()
        self._ck(self.L.pg_search_status(self.h, C.byref(a), C.byref(b), C.byref(r)))
        return a.value, b.value, r.as_dict()

    def search_lookup(self, pos):
        a = np.ascontiguousarray(pos, dtype=np.uint16)
        f, g, p = C.c_int32(), C.c_int32(), C.c_int32()
        self._ck(self.L.pg_search_lookup(self.h, a.ctypes.data, C.byref(f), C.byref(g), C.byref(p)))
        return (g.value, p.value) if f.value else None

    def search_end(self):
        self._ck(self.L.pg_search_end(self.h))

    def xrec_stride(self):
        return self.L.pg_xrec_stride(self.h)
