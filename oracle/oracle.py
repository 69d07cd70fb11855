"""ctypes binding of oracle/libpastar_oracle.so (plain-C restatement).

TEST INFRASTRUCTURE — see pastar_oracle.h for the parity-pinning statement.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libpastar_oracle.so")
MAX_SEQ = 16
HASH = {"FZORDER": 0, "PZORDER": 1, "FSUM": 2, "PSUM": 3}


class Succ(C.Structure):
    _fields_ = [("pos", C.c_uint16 * MAX_SEQ), ("f", C.c_int32), ("g", C.c_int32), ("parenti", C.c_int32),
                ("owner", C.c_uint32)]


class SearchResult(C.Structure):
    _fields_ = [("finished", C.c_int32), ("g", C.c_int32), ("f", C.c_int32), ("pops", C.c_int64),
                ("expansions", C.c_int64), ("generated", C.c_int64), ("reopen", C.c_int64),
                ("open_size", C.c_int64), ("closed_size", C.c_int64)]


def build():
    """Compile the C restatement (gcc only; no reference sources involved)."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(os.path.join(_HERE, "pastar_oracle.c")):
            build()
        L = C.CDLL(_LIB)
        L.po_cost_table.argtypes = [C.c_void_p]
        L.po_pair_table.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p]
        L.po_weights.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.c_void_p]
        L.po_weights.restype = C.c_int
        L.po_create.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.c_void_p]
        L.po_create.restype = C.c_void_p
        L.po_destroy.argtypes = [C.c_void_p]
        L.po_table.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.po_table.restype = C.POINTER(C.c_int32)
        L.po_int_weights.argtypes = [C.c_void_p]
        L.po_int_weights.restype = C.POINTER(C.c_int32)
        L.po_calculate_h.argtypes = [C.c_void_p, C.c_void_p]
        L.po_calculate_h.restype = C.c_int32
        L.po_owner.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.po_owner.restype = C.c_uint32
        L.po_get_neigh.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(Succ)]
        L.po_get_neigh.restype = C.c_int
        L.po_astar.argtypes = [C.c_void_p, C.c_int64, C.POINTER(SearchResult), C.POINTER(C.c_char_p)]
        L.po_astar.restype = C.c_int
        L.po_astar_settled.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.POINTER(SearchResult)]
        L.po_astar_settled.restype = C.c_int64
        _lib = L
    return _lib


def _seq_args(seqs):
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    arr = (C.c_char_p * len(bs))(*bs)
    lens = (C.c_int * len(bs))(*[len(b) for b in bs])
    return bs, arr, lens


def cost_table():
    out = np.zeros(90 * 90, dtype=np.int32)
    lib().po_cost_table(out.ctypes.data)
    return out.reshape(90, 90)


def pair_table(s1, s2):
    b1, b2 = s1.encode(), s2.encode()
    out = np.zeros((len(b1) + 1, len(b2) + 1), dtype=np.int32)
    lib().po_pair_table(b1, len(b1), b2, len(b2), out.ctypes.data)
    return out


def weights(seqs):
    bs, arr, lens = _seq_args(seqs)
    n = len(bs)
    out = np.zeros((n, n), dtype=np.float32)
    rc = lib().po_weights(n, arr, lens, out.ctypes.data)
    if rc != 0:
        raise ValueError("sequence longer than the reference weight routine supports (998)")
    return out


# successor records as a structured array: the common currency of the parity tests
def succ_dtype(n):
    return np.dtype([("pos", np.uint16, (n,)), ("f", np.int32), ("g", np.int32), ("parenti", np.int32),
                     ("owner", np.uint32)])


class Problem:
    """Sequences + P reverse-DP tables + truncated int weights (HeuristicHPair.cpp:47-67)."""

    def __init__(self, seqs, w_int=None):
        self.seqs = [s if isinstance(s, str) else s.decode() for s in seqs]
        self.n = len(seqs)
        self._keep = _seq_args(seqs)
        wp = None
        if w_int is not None:
            self._w = np.ascontiguousarray(w_int, dtype=np.int32).reshape(self.n, self.n)
            wp = self._w.ctypes.data
        self.h = lib().po_create(self.n, self._keep[1], self._keep[2], wp)
        if not self.h:
            raise ValueError("po_create failed")
        self.npairs = self.n * (self.n - 1) // 2

    def close(self):
        if self.h:
            lib().po_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def lens(self):
        return [len(s) for s in self.seqs]

    def int_weights(self):
        p = lib().po_int_weights(self.h)
        return np.ctypeslib.as_array(p, shape=(self.n * self.n,))[: self.n * self.n].reshape(self.n, self.n).copy()

    def table(self, pair):
        r, c = C.c_int(), C.c_int()
        p = lib().po_table(self.h, pair, C.byref(r), C.byref(c))
        return np.ctypeslib.as_array(p, shape=(r.value * c.value,)).reshape(r.value, c.value)

    def calculate_h(self, pos):
        a = np.ascontiguousarray(pos, dtype=np.uint16)
        return int(lib().po_calculate_h(self.h, a.ctypes.data))

    def get_neigh(self, pos, g, parenti, vec_size=1, hash_type="FZORDER", shift=12):
        a = np.ascontiguousarray(pos, dtype=np.uint16)
        buf = (Succ * ((1 << self.n) - 1))()
        cnt = lib().po_get_neigh(self.h, a.ctypes.data, int(g), int(parenti), vec_size, HASH[hash_type], shift, buf)
        out = np.zeros(cnt, dtype=succ_dtype(self.n))
        for k in range(cnt):
            out["pos"][k] = buf[k].pos[: self.n]
            out["f"][k], out["g"][k], out["parenti"][k], out["owner"][k] = buf[k].f, buf[k].g, buf[k].parenti, buf[k].owner
        return out

    def astar(self, budget=0, want_rows=True):
        res = SearchResult()
        rows = None
        if want_rows:
            total = sum(self.lens) + 1
            bufs = [C.create_string_buffer(total) for _ in range(self.n)]
            rows = (C.c_char_p * self.n)(*[C.cast(b, C.c_char_p) for b in bufs])
        lib().po_astar(self.h, budget, C.byref(res), rows)
        d = {k: getattr(res, k) for k, _ in SearchResult._fields_}
        if want_rows and res.finished:
            d["rows"] = [b.value.decode() for b in bufs]
        return d

    def astar_settled(self, budget=0, cap=None):
        """The serial A* of astar() for `budget` pops (0: to the goal), then its settled set: (F, pos, g, parenti), where
        F is the f of the best live open entry and pos[k] / g[k] / parenti[k] are the closed nodes with f < F."""
        if cap is None:
            cap = budget + 1 if budget > 0 else 1 << 16
        while True:
            pos = np.zeros((cap, self.n), dtype=np.uint16)
            g = np.zeros(cap, dtype=np.int32)
            par = np.zeros(cap, dtype=np.int32)
            F, res = C.c_int32(), SearchResult()
            k = lib().po_astar_settled(self.h, budget, cap, C.byref(F), pos.ctypes.data, g.ctypes.data, par.ctypes.data,
                                       C.byref(res))
            if k <= cap:
                return F.value, pos[:k], g[:k], par[:k]
            cap = k


def owner(pos, hash_type="FZORDER", shift=12, size=1):
    a = np.ascontiguousarray(pos, dtype=np.uint16)
    return int(lib().po_owner(a.shape[-1], a.ctypes.data, HASH[hash_type], shift, size))
